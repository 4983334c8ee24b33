"""Argument errors of the eleven frame-batched entry points of d3d_b200.box, in both call forms, raised before any device work: every
call below runs with _cabi.to_device and _cabi.require_cuda replaced by a function that raises DeviceWork, which none of the expected
exceptions catches.  Needs no GPU."""
import numpy as np
import pytest

import d3d_b200.box as B
from d3d_b200 import _cabi


class DeviceWork(Exception):
    pass


@pytest.fixture(autouse=True)
def no_device(monkeypatch):
    def touched(*a, **k):
        raise DeviceWork("device work before the argument checks")
    monkeypatch.setattr(_cabi, "to_device", touched)
    monkeypatch.setattr(_cabi, "require_cuda", touched)


def _rows(n, k, dt=np.float64):
    return (np.random.default_rng(n).random((n, k)) + .5).astype(dt)


class Pair:
    """an entry point over two per-frame sets of `ka` / `kb` columns: fn(a, b, offsets_a, offsets_b, **kw).  `columns`: the message
    fragments of a wrong column count in the first and in the second set; `axis`: takes project_axis; `cross`: None if mixed dtypes are
    cast, else the arguments under which two sets of different dtypes raise"""
    def __init__(self, fn, ka, kb, columns, axis=False, cross=None, **kw):
        self.fn, self.ka, self.kb, self.kw = fn, ka, kb, kw
        self.columns, self.axis, self.cross = columns, axis, cross

    def lists(self, na, nb, ka=None, kb=None, dts=(np.float64, np.float64), **kw):
        la = [_rows(n, ka or self.ka, dt) for n, dt in zip(na, dts)]
        return self.fn(la, [_rows(m, kb or self.kb) for m in nb], **{**self.kw, **kw})

    def packed(self, oa, ob):
        return self.fn(_rows(9, self.ka), _rows(7, self.kb), oa, ob, **self.kw)

    def no_offsets(self):
        return self.fn(_rows(9, self.ka), _rows(7, self.kb), **self.kw)


class Nms:
    """box2d_nms_batch: one set of frames carrying boxes [n_f, 5] and scores [n_f].  It takes one set of offsets: where the
    column offsets of a packed call hold another number of frames, the call gets one score too few instead.  Boxes are read as rows of
    5 values, so rows of another width make another number of boxes than of scores; mixed dtypes promote"""
    columns, axis, cross = ("inconsistent", None), False, None

    def lists(self, na, nb, ka=5):
        return B.box2d_nms_batch([_rows(n, ka) for n in na], [_rows(m, 1)[:, 0] for m in nb])

    def packed(self, oa, ob):
        return B.box2d_nms_batch(_rows(9, 5), _rows(9 if len(ob) == len(oa) else 8, 1)[:, 0], oa)

    def no_offsets(self):
        return B.box2d_nms_batch(_rows(9, 5), _rows(9, 1)[:, 0])


class Match:
    """match_greedy_batch: a [n_f, m_f] distance block per frame, n_f scores and source tags, m_f destination tags"""
    columns, axis, cross = ("NxM", None), False, None   # distances are cast to float32
    thr = np.full(2, .5, np.float32)

    def lists(self, na, nb, ka=None):
        dist = [_rows(n, m, np.float32) if ka is None else _rows(n * m, 1, np.float32)[:, 0] for n, m in zip(na, nb)]
        return B.match_greedy_batch(dist, [_rows(n, 1)[:, 0] for n in na], [np.zeros(n, np.int32) for n in na],
                                    [np.zeros(m, np.int32) for m in nb], self.thr)

    def _packed(self, *offsets):
        blk = np.array([0, 4 * 3, 4 * 3 + 5 * 4])   # the blocks of frames of 4 x 3 and 5 x 4
        return B.match_greedy_batch((_rows(32, 1, np.float32)[:, 0], blk), _rows(9, 1)[:, 0], np.zeros(9, np.int32), np.zeros(7, np.int32), self.thr,
                                    *offsets)

    def packed(self, oa, ob):
        return self._packed(oa, ob)

    def no_offsets(self):   # taken as the list form of two frames, (distances, block offsets), whose scores and tags do not match
        return self._packed()


ENTRIES = {
    "box2d_iou_batch": Pair(B.box2d_iou_batch, 5, 5, ("fields", "fields"), cross=dict(precise=False)),
    "box2d_iou_max_batch": Pair(B.box2d_iou_max_batch, 5, 5, ("fields", "fields"), cross=dict(precise=False)),
    "box2d_nms_batch": Nms(),
    "box2dr_crop_batch": Pair(B.box2dr_crop_batch, 2, 5, ("Nx2", "5 fields"), cross={}),
    "box3dp_crop_batch": Pair(B.box3dp_crop_batch, 3, 7, ("Nx3", "7 fields"), axis=True, cross={}),
    "box2dr_crop_assign_batch": Pair(B.box2dr_crop_assign_batch, 2, 5, ("Nx2", "5 fields"), cross={}),
    "box3dp_crop_assign_batch": Pair(B.box3dp_crop_assign_batch, 3, 7, ("Nx3", "7 fields"), axis=True, cross={}),
    "box2dr_pdist_batch": Pair(B.box2dr_pdist_batch, 2, 5, ("Nx2", "5 fields"), cross={}),
    "box3dr_pdist_batch": Pair(B.box3dr_pdist_batch, 3, 7, ("Nx3", "7 fields"), axis=True, cross={}),
    "box3d_iou_distance_batch": Pair(B.box3d_iou_distance_batch, 7, 7, ("Nx7", "Nx7")),
    "match_greedy_batch": Match(),
}
ENTRY = pytest.mark.parametrize("name", list(ENTRIES))


@ENTRY
def test_empty_list(name):
    e = ENTRIES[name]
    assert e.lists([], []) == []


@ENTRY
def test_frame_counts_differ(name):
    with pytest.raises(ValueError):
        ENTRIES[name].lists([4, 5], [3])


@ENTRY
def test_packed_without_offsets(name):
    with pytest.raises(ValueError):
        ENTRIES[name].no_offsets()


@ENTRY
def test_offsets_not_ascending(name):
    e = ENTRIES[name]
    with pytest.raises(ValueError, match="ascending"):
        e.packed(np.array([2, 6, 9]), np.array([0, 3, 7]))    # the first 2 rows in no frame
    with pytest.raises(ValueError, match="ascending"):
        e.packed(np.array([0, 6, 4, 9]), np.array([0, 2, 5, 7]))


@ENTRY
def test_offsets_disagree_with_rows(name):
    e = ENTRIES[name]
    with pytest.raises(ValueError):
        e.packed(np.array([0, 4, 8]), np.array([0, 3, 7]))    # 8 rows of 9
    with pytest.raises(ValueError):
        e.packed(np.array([0, 4, 9]), np.array([0, 7]))       # 2 frames of rows, 1 of columns


@pytest.mark.parametrize("name,side", [(n, side) for n, e in ENTRIES.items() for side in (0, 1) if e.columns[side]])
def test_wrong_columns(name, side):
    e = ENTRIES[name]
    if isinstance(e, Pair):
        bad = dict(ka=e.ka + 1) if side == 0 else dict(kb=e.kb + 1)
    else:   # box2d_nms_batch: frames of 5 and 10 boxes of 6 values make 18 rows of 5 for 15 scores; match_greedy_batch: 1-D distances
        bad = dict(ka=6 if isinstance(e, Nms) else 1)
    with pytest.raises(ValueError, match=e.columns[side]):
        e.lists([5, 10], [5, 10], **bad)


@pytest.mark.parametrize("name", [n for n, e in ENTRIES.items() if e.axis])
def test_project_axis(name):
    e = ENTRIES[name]
    for ax in (3, -1):
        with pytest.raises(ValueError, match="projection axis"):
            e.lists([4, 5], [3, 4], project_axis=ax)


@pytest.mark.parametrize("name", [n for n, e in ENTRIES.items() if e.cross is not None])
def test_mixed_dtypes(name):
    e = ENTRIES[name]
    with pytest.raises(RuntimeError, match="same dtype"):   # within a set
        e.lists([4, 5], [3, 4], dts=(np.float32, np.float64))
    with pytest.raises(RuntimeError, match="same dtype"):   # float32 rows, float64 columns
        e.lists([4, 5], [3, 4], dts=(np.float32, np.float32), **e.cross)
