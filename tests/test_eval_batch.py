"""Frame-batched detection matching (box3d_iou_distance_batch / d3d_iou3d_distance_batch_f32, match_greedy_batch /
d3d_match_greedy_batch_f32): per frame the distance block equals box3d_iou_distance bit for bit, and per frame and threshold set the
assignment equals match_greedy."""
import ctypes as C

import numpy as np
import pytest
import torch

from conftest import golden
from d3d_b200 import _cabi


def _boxes3d(rng, n, extent=40.0, shift=0.0):
    return np.stack([(rng.random(n) - .5) * extent + shift, (rng.random(n) - .5) * extent + shift, rng.normal(-1, 0.5, n),
                     3.5 + rng.random(n) * 2, 1.5 + rng.random(n), 1.4 + rng.random(n) * 0.6, (rng.random(n) - .5) * 7], 1).astype(np.float32)


def _frame(rng, n, m, shift=0.0):
    """n detections, m ground-truth boxes; a third of the detections sit on a ground-truth box"""
    gt, dt = _boxes3d(rng, m, shift=shift), _boxes3d(rng, n, shift=shift)
    k = min(n, m) // 3 if m else 0
    if k:
        dt[:k] = gt[rng.integers(0, m, k)] + rng.normal(0, 0.2, (k, 7)).astype(np.float32)
    return dt, gt


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda:0")


def _t(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def _bits(x):
    return np.ascontiguousarray(x.cpu().numpy() if torch.is_tensor(x) else x).view(np.uint32)


# ------------------------------------------------------------------ C ABI, no GPU needed
def test_cabi_argument_errors_without_gpu():
    """argument errors return codes before any CUDA call"""
    lib = C.CDLL(_cabi.LIB_PATH)
    i64, vp, sz = C.c_int64, C.c_void_p, C.c_size_t
    wsb = lib.d3d_iou3d_distance_batch_workspace_bytes
    wsb.restype, wsb.argtypes = sz, [i64, i64, i64]
    dist = lib.d3d_iou3d_distance_batch_f32
    dist.argtypes = [vp, i64, vp, vp, i64, vp, i64, i64, i64, C.c_int, vp, vp, vp, sz, vp]
    need = wsb(10, 20, 3)
    assert need >= (10 + 3 * 64) * 32 + (20 + 3 * 128) * 32 and wsb(-1, 20, 3) == 0
    ok = (8, 10, 8, 8, 20, 8, 3, 5, 9, 1, 8, 8, 8, need, 0)

    def call(**kw):
        a = list(ok)
        for k, v in kw.items():
            a[["b1", "t1", "o1", "b2", "t2", "o2", "nf", "mx1", "mx2", "rot", "do", "d", "ws", "wsb", "st"].index(k)] = v
        return dist(*a)

    assert call(t1=-1) == _cabi.ERR_INVALID and call(t2=-1) == _cabi.ERR_INVALID and call(nf=-1) == _cabi.ERR_INVALID
    assert call(mx1=-1) == _cabi.ERR_INVALID and call(mx2=-1) == _cabi.ERR_INVALID
    assert call(nf=0) == _cabi.OK and call(t1=0) == _cabi.OK and call(t2=0) == _cabi.OK   # every block empty: no-op
    assert call(wsb=need - 1) == _cabi.ERR_WORKSPACE and call(ws=0) == _cabi.ERR_WORKSPACE
    assert call(rot=0, wsb=need - 1) == _cabi.ERR_WORKSPACE
    assert call(o1=0) == _cabi.ERR_INVALID and call(do=0) == _cabi.ERR_INVALID
    assert call(mx1=64 * 65536) == _cabi.ERR_UNSUPPORTED and call(mx2=128 * 65536) == _cabi.ERR_UNSUPPORTED   # more than 65535 tiles

    mg = lib.d3d_match_greedy_batch_f32
    mg.argtypes = [vp, vp, vp, vp, i64, i64, vp, vp, vp, vp, C.c_int32, C.c_int32, vp, vp, vp]
    mok = (8, 8, 8, 8, 3, 40, 8, 8, 8, 8, 40, 3, 8, 8, 0)

    def mcall(**kw):
        a = list(mok)
        for k, v in kw.items():
            a[["d", "do", "so", "o", "nf", "mx", "ord", "st", "dt", "thr", "ns", "nc", "sa", "da", "stream"].index(k)] = v
        return mg(*a)

    assert mcall(nf=-1) == _cabi.ERR_INVALID and mcall(mx=-1) == _cabi.ERR_INVALID and mcall(ns=-1) == _cabi.ERR_INVALID
    assert mcall(nc=0) == _cabi.ERR_INVALID
    assert mcall(mx=4097) == _cabi.ERR_UNSUPPORTED and mcall(mx=4097, nf=0) == _cabi.ERR_UNSUPPORTED
    assert mcall(nf=0) == _cabi.OK and mcall(ns=0) == _cabi.OK
    assert mcall(thr=0) == _cabi.ERR_INVALID and mcall(ord=0) == _cabi.ERR_INVALID


# ------------------------------------------------------------------ distance matrix
def _check_dist_per_frame(frames, metric, dev, sample=None):
    from d3d_b200.box import box3d_iou_distance, box3d_iou_distance_batch
    blocks = box3d_iou_distance_batch([_t(a, dev) for a, _ in frames], [_t(b, dev) for _, b in frames], metric=metric)
    assert len(blocks) == len(frames)
    for f in (range(len(frames)) if sample is None else sample):
        a, b = frames[f]
        blk = blocks[f]
        assert blk.is_cuda and blk.dtype == torch.float32 and tuple(blk.shape) == (len(a), len(b)), f
        single = box3d_iou_distance(_t(a, dev), _t(b, dev), metric)
        assert np.array_equal(_bits(blk), _bits(single)), (metric, f, len(a), len(b))
    return blocks


@pytest.mark.gpu
@pytest.mark.parametrize("metric", ["riou", "iou"])
def test_distance_batch_bit_equal_per_frame(dev, metric):
    """ragged frames: empty on either side, 1 x 1, the tile edges 63/64/65 rows x 127/128/129 columns, several hundred by several
    hundred, a frame 3e5 m from the origin, and the golden dist3d inputs packed between two other frames"""
    rng = np.random.default_rng(17)
    g = golden("dist3d.npz")
    sizes = [(0, 7), (9, 0), (0, 0), (1, 1), (63, 127), (64, 128), (65, 129), (40, 12), (450, 380), (2, 300)]
    frames = [_frame(rng, n, m) for n, m in sizes]
    frames.insert(5, _frame(rng, 70, 50, shift=3e5))
    frames += [_frame(rng, 150, 40), (g["src"], g["dst"]), _frame(rng, 33, 65)]
    blocks = _check_dist_per_frame(frames, metric, dev)
    assert (blocks[9] < 0.5).any() and (blocks[5] < 0.5).any()   # real overlaps, not only the constant 1 of rejected pairs


@pytest.mark.gpu
@pytest.mark.parametrize("metric", ["riou", "iou"])
def test_distance_batch_over_65535_frames(dev, metric):
    """70 000 frames of 1-3 boxes each: frames on grid.x beyond 65 535"""
    rng = np.random.default_rng(23)
    nf = 70000
    ns, ms = rng.integers(1, 4, nf), rng.integers(1, 4, nf)
    A, B = _boxes3d(rng, int(ns.sum()), extent=6.0), _boxes3d(rng, int(ms.sum()), extent=6.0)
    oa, ob = np.cumsum(np.r_[0, ns]), np.cumsum(np.r_[0, ms])
    frames = [(A[oa[f]:oa[f + 1]], B[ob[f]:ob[f + 1]]) for f in range(nf)]
    sample = list(range(0, nf, 499)) + list(range(65530, 65541)) + list(range(nf - 150, nf))
    blocks = _check_dist_per_frame(frames, metric, dev, sample)
    assert sum(bool((blocks[f] < 1).any()) for f in sample) > len(sample) // 4


# ------------------------------------------------------------------ matching
THR40 = np.stack([np.array([0.3, 0.5, 0.6]) + t for t in np.linspace(0.0, 0.65, 40)]).astype(np.float32)   # 40 sets x 3 categories


def _match_frames(rng, sizes, dev, odd_tags=True, ties=True):
    """per-frame (distance, scores, src tags, dst tags): distances from the distance kernel, then tied values, NaN distances, tied and
    NaN scores, and tags -1 and >= 3 (outside the 3 categories)"""
    from d3d_b200.box import box3d_iou_distance
    out = []
    for i, (n, m) in enumerate(sizes):
        a, b = _frame(rng, n, m)
        d = box3d_iou_distance(a, b, "riou")
        s = rng.random(n)
        st, dt = rng.integers(0, 3, n).astype(np.int32), rng.integers(0, 3, m).astype(np.int32)
        if ties and n and m:
            d[rng.random((n, m)) < 0.05] = np.nan
            q = rng.random((n, m)) < 0.3
            d[q] = np.round(d[q] * 8) / 8          # tied distances inside a row
            s = np.round(s * 10) / 10              # tied scores
            s[rng.random(n) < 0.05] = np.nan
        if odd_tags and n and m:
            st[rng.random(n) < 0.08] = -1
            st[rng.random(n) < 0.05] = 3
            dt[rng.random(m) < 0.05] = 7
            dt[rng.random(m) < 0.05] = -1
        out.append((d, s, st, dt))
    return out


def _check_match_per_frame(frames, thr, dev):
    from d3d_b200.box import match_greedy, match_greedy_batch
    res = match_greedy_batch([_t(d, dev) for d, *_ in frames], [_t(s, dev) for _, s, _, _ in frames], [_t(x, dev) for *_, x, _ in frames],
                             [_t(x, dev) for *_, x in frames], _t(thr, dev))
    assert len(res) == len(frames)
    T = len(thr) if thr.ndim == 2 else None
    for (d, s, st, dt), (sa, da) in zip(frames, res):
        assert sa.is_cuda and sa.dtype == torch.int32 and da.dtype == torch.int32
        assert tuple(sa.shape) == ((T, len(s)) if T else (len(s),)) and tuple(da.shape) == ((T, len(dt)) if T else (len(dt),))
        es, ed = match_greedy(_t(d, dev), _t(s, dev), _t(st, dev), _t(dt, dev), _t(thr, dev))
        assert torch.equal(sa, es) and torch.equal(da, ed), (d.shape, int((sa != es).sum()), int((da != ed).sum()))
    return res


@pytest.mark.gpu
def test_match_batch_equals_per_frame(dev):
    """40 threshold sets, 3 categories; frames without sources or destinations; tags -1 and >= ncat; tied and NaN scores and distances"""
    rng = np.random.default_rng(29)
    sizes = [(150, 40), (0, 30), (25, 0), (0, 0), (1, 1), (300, 64), (64, 300), (7, 129), (170, 45), (500, 1000), (33, 2)]
    frames = _match_frames(rng, sizes, dev)
    res = _check_match_per_frame(frames, THR40, dev)
    assert sum(int((sa >= 0).sum()) for sa, _ in res) > 1000   # many matches, not only -1
    _check_match_per_frame(frames, THR40[17], dev)              # one set: the leading dimension is dropped
    _check_match_per_frame(_match_frames(rng, sizes, dev, odd_tags=False, ties=False), THR40, dev)


@pytest.mark.gpu
def test_match_batch_vs_oracle(dev, oracle):
    """small frames against the restated walk of the reference (tags inside [0, ncat), which the restatement indexes thresholds with)"""
    from d3d_b200.box import match_greedy_batch
    rng = np.random.default_rng(31)
    frames = _match_frames(rng, [(12, 9), (30, 20), (5, 40), (1, 1), (60, 45)], dev, odd_tags=False)
    res = match_greedy_batch([d for d, *_ in frames], [s for _, s, _, _ in frames], [x for *_, x, _ in frames], [x for *_, x in frames], THR40)
    for (d, s, st, dt), (sa, da) in zip(frames, res):
        assert isinstance(sa, np.ndarray)
        for t in (0, 9, 22, 39):
            osa, oda = oracle.match_greedy(d, s, st, dt, THR40[t])
            assert np.array_equal(sa[t], osa) and np.array_equal(da[t], oda), (d.shape, t)


@pytest.mark.gpu
def test_match_batch_fallback_over_4096_destinations(dev):
    """a frame of 5000 destinations: every frame takes one match_greedy call"""
    rng = np.random.default_rng(37)
    frames = _match_frames(rng, [(80, 30), (200, 5000), (0, 4097), (40, 12)], dev)
    _check_match_per_frame(frames, THR40, dev)


@pytest.mark.gpu
def test_call_forms(dev):
    """list and packed forms agree; numpy in -> numpy out; host tensors in -> host tensors out"""
    from d3d_b200.box import box3d_iou_distance_batch, match_greedy_batch
    rng = np.random.default_rng(43)
    sizes = [(150, 40), (0, 12), (65, 129), (9, 0), (30, 31)]
    fr = [_frame(rng, n, m) for n, m in sizes]
    so, do = np.cumsum([0] + [n for n, _ in sizes]), np.cumsum([0] + [m for _, m in sizes])
    A, B = np.concatenate([a for a, _ in fr]), np.concatenate([b for _, b in fr])
    scores, st, dt = rng.random(len(A)), rng.integers(0, 3, len(A)).astype(np.int32), rng.integers(0, 3, len(B)).astype(np.int32)

    lst = box3d_iou_distance_batch([_t(a, dev) for a, _ in fr], [_t(b, dev) for _, b in fr])
    flat, doff = box3d_iou_distance_batch(_t(A, dev), _t(B, dev), torch.from_numpy(so), torch.from_numpy(do))
    assert flat.is_cuda and doff.device.type == "cpu" and doff.tolist() == np.cumsum([0] + [n * m for n, m in sizes]).tolist()
    assert np.array_equal(_bits(flat), _bits(torch.cat([x.reshape(-1) for x in lst])))
    assert all(x.untyped_storage().data_ptr() == lst[0].untyped_storage().data_ptr() for x in lst)   # views into one buffer
    flat_np, doff_np = box3d_iou_distance_batch(A, B, so, do, metric="riou")
    assert isinstance(flat_np, np.ndarray) and isinstance(doff_np, np.ndarray) and np.array_equal(_bits(flat_np), _bits(flat))
    lst_np = box3d_iou_distance_batch([a for a, _ in fr], [b for _, b in fr])
    assert all(isinstance(x, np.ndarray) and x.shape == (n, m) for x, (n, m) in zip(lst_np, sizes))
    flat_cpu, _ = box3d_iou_distance_batch(torch.from_numpy(A), torch.from_numpy(B), so, do)
    assert flat_cpu.device.type == "cpu" and np.array_equal(_bits(flat_cpu), _bits(flat))
    assert box3d_iou_distance_batch([], []) == []
    f0, o0 = box3d_iou_distance_batch(torch.zeros((0, 7)), torch.zeros((0, 7)), [0], [0])
    assert f0.numel() == 0 and o0.tolist() == [0]
    with pytest.raises(ValueError):
        box3d_iou_distance_batch([torch.zeros((3, 5))], [torch.zeros((3, 7))])
    with pytest.raises(ValueError):
        box3d_iou_distance_batch(A, B, so, do, metric="giou")
    with pytest.raises(ValueError):
        box3d_iou_distance_batch(A, B, so[:-1], do[:-1])
    with pytest.raises(ValueError):
        box3d_iou_distance_batch(A, B)

    sl = [scores[so[f]:so[f + 1]] for f in range(len(sizes))]
    tl, ul = [st[so[f]:so[f + 1]] for f in range(len(sizes))], [dt[do[f]:do[f + 1]] for f in range(len(sizes))]
    ml = match_greedy_batch(lst, [_t(x, dev) for x in sl], [_t(x, dev) for x in tl], [_t(x, dev) for x in ul], _t(THR40, dev))
    sa, da = match_greedy_batch((flat, doff), _t(scores, dev), _t(st, dev), _t(dt, dev), _t(THR40, dev), torch.from_numpy(so), torch.from_numpy(do))
    assert sa.is_cuda and tuple(sa.shape) == (40, len(A)) and tuple(da.shape) == (40, len(B))
    assert torch.equal(sa, torch.cat([x for x, _ in ml], 1)) and torch.equal(da, torch.cat([y for _, y in ml], 1))
    sa_np, da_np = match_greedy_batch((flat_np, doff_np), scores, st, dt, THR40, so, do)
    assert isinstance(sa_np, np.ndarray) and np.array_equal(sa_np, sa.cpu().numpy()) and np.array_equal(da_np, da.cpu().numpy())
    sa_cpu, da_cpu = match_greedy_batch((flat_cpu, doff), torch.from_numpy(scores), torch.from_numpy(st), torch.from_numpy(dt), torch.from_numpy(THR40),
                                        so, do)
    assert sa_cpu.device.type == "cpu" and torch.equal(sa_cpu, sa.cpu()) and torch.equal(da_cpu, da.cpu())
    s1, d1 = match_greedy_batch((flat, doff), scores, st, dt, THR40[3], so, do)   # one set: [total]
    assert tuple(s1.shape) == (len(A),) and torch.equal(s1, sa[3]) and torch.equal(d1, da[3])
    ml_np = match_greedy_batch(lst_np, sl, tl, ul, THR40[3])
    assert all(isinstance(x, np.ndarray) and np.array_equal(x, sa[3, so[f]:so[f + 1]].cpu().numpy()) for f, (x, _) in enumerate(ml_np))
    assert match_greedy_batch([], [], [], [], THR40) == []
    with pytest.raises(ValueError):
        match_greedy_batch((flat, doff), scores[:-1], st[:-1], dt, THR40, so, do)
    with pytest.raises(ValueError):
        match_greedy_batch((flat[:-1], doff), scores, st, dt, THR40, so, do)
    with pytest.raises(ValueError):
        match_greedy_batch(lst, sl, tl, ul[:-1], THR40)
    torch.cuda.synchronize()
