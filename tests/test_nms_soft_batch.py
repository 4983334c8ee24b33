"""Frame-batched soft-NMS (box2d_nms_batch with supression_method 'linear' / 'gaussian', d3d_nms2d_batch_soft_*): per frame the keep
mask of box2d_nms with the same arguments, bit for bit, and the reference's own masks on the soft-NMS fixtures."""
import numpy as np
import pytest
import torch

from conftest import golden, gen_boxes, proposals, SOFT_CASES, SOFT_TEST6, soft_inputs
from d3d_b200 import _cabi

pytestmark = pytest.mark.gpu

PARAM = {"linear": 1.0, "gaussian": 0.5}


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda:0")


def _t(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def _frames(rng, sizes, ties=()):
    out = []
    for n in sizes:
        if n == 0:
            out.append((np.zeros((0, 5)), np.zeros(0)))
            continue
        b, s = proposals(rng, n, max(n // 25, 1), extent=30.0)
        if n in ties:
            s = np.round(s * 20) / 20   # tied scores: the stable order puts the lower index first
        out.append((b, s))
    return out


def _check_per_frame(dev, frames, im, m, thr, sthr, precise, dtype):
    from d3d_b200.box import box2d_nms, box2d_nms_batch
    bl = [_t(b.astype(dtype), dev) for b, _ in frames]
    sl = [_t(s.astype(dtype), dev) for _, s in frames]
    keeps = box2d_nms_batch(bl, sl, iou_method=im, iou_threshold=thr, score_threshold=sthr, precise=precise,
                            supression_method=m, supression_param=PARAM[m])
    assert len(keeps) == len(frames)
    for b, s, k in zip(bl, sl, keeps):
        assert k.dtype == torch.bool and k.shape == (len(b),)
        if len(b):
            single = box2d_nms(b, s, im, m, iou_threshold=thr, score_threshold=sthr, supression_param=PARAM[m], precise=precise)
            assert torch.equal(k, single), (im, m, thr, sthr, precise, len(b), int((k != single).sum()))


@pytest.mark.parametrize("im", ["box", "rbox"])
@pytest.mark.parametrize("m", ["linear", "gaussian"])
def test_batch_equals_per_frame(dev, im, m):
    """ragged frames (empty, one box, 64, 65, tied scores, 4096, 8192), fp64 and fp32, thresholds 0, 0.3 and -1, score threshold 0 and
    0.2.  Under a negative threshold every pair decays and every step re-sorts the whole range: those frames stay small (the per-frame
    calls alone would take minutes on the large ones)."""
    rng = np.random.default_rng(5)
    big = _frames(rng, (700, 0, 1, 64, 4096, 65, 1500, 8192), ties=(1500,))
    small = _frames(rng, (300, 0, 1, 64, 65, 1500), ties=(300,))
    for precise, dtype in ((True, np.float64), (False, np.float32)):
        for thr in (0.0, 0.3, -1.0):
            for sthr in (0.0, 0.2):
                _check_per_frame(dev, small if thr < 0 else big, im, m, thr, sthr, precise, dtype)


@pytest.mark.parametrize("im", ["box", "rbox"])
@pytest.mark.parametrize("m", ["linear", "gaussian"])
@pytest.mark.parametrize("case", ["above", "negative"])
def test_batch_equals_per_frame_running_S(dev, im, m, case):
    """the regimes of the running end S of the re-sort range.  'above': every score above the score threshold (proposals filtered
    before soft-NMS), so no box starts suppressed, S starts at none in the middle of the frame and grows with every box the decay
    suppresses.  'negative': scores in [-1, 1) and a negative score threshold, so a decay can lift a suppressed box back over the
    threshold and S is found again by a scan.  Both must move the keep mask away from `score > score_threshold`: the decay and the
    re-sort decide it."""
    from d3d_b200.box import box2d_nms_batch
    rng = np.random.default_rng(41)
    frames = _frames(rng, (700, 0, 65, 1500, 4096))
    sthr = 0.45 if case == "above" else -0.3
    frames = [(b, 0.5 + 0.5 * s / 1.1 if case == "above" else 2.0 * s / 1.1 - 1.0) for b, s in frames]   # proposals' scores: [0, 1.1)
    for precise, dtype in ((True, np.float64), (False, np.float32)):
        for thr in (0.0, 0.3):
            _check_per_frame(dev, frames, im, m, thr, sthr, precise, dtype)
            keeps = box2d_nms_batch([b for b, _ in frames], [s for _, s in frames], iou_method=im, iou_threshold=thr, score_threshold=sthr,
                                    supression_method=m, supression_param=PARAM[m])
            moved = [bool((k != (s > sthr)).any()) for (_, s), k in zip(frames, keeps) if len(s) >= 65]
            if case == "above":
                assert all(moved), (im, m, thr, moved)   # boxes suppressed by the decay alone
            else:
                assert any(moved), (im, m, thr)         # suppressed boxes lifted back over the threshold and kept
                assert all(((s > sthr) <= k).all() for (_, s), k in zip(frames, keeps))   # a decay never suppresses a box above -0.3 here


def test_fixtures_packed_between_frames(dev):
    """every soft-NMS fixture input, packed as the middle frame of three, gives the reference's own mask (nms_soft.npz)"""
    from d3d_b200.box import box2d_nms_batch
    g = golden("nms_soft.npz")
    rng = np.random.default_rng(9)
    (fb0, fs0), (fb1, fs1) = _frames(rng, (300, 1000))

    def middle(b, s, **kw):
        off = np.cumsum([0, len(fb0), len(b), len(fb1)])
        keep = box2d_nms_batch(_t(np.concatenate([fb0, b, fb1]), dev), _t(np.concatenate([fs0, s, fs1]), dev), torch.from_numpy(off), **kw)
        return keep.cpu().numpy()[off[1]:off[2]]

    nb, ns = SOFT_TEST6
    for m in ("linear", "gaussian"):
        for im in ("box", "rbox"):
            keep = middle(nb, ns, iou_method=im, iou_threshold=0.1, score_threshold=0.15, supression_method=m, supression_param=PARAM[m])
            assert np.array_equal(keep, g[f"test6_{m}_{im}"]), (m, im)
    for tag, n, gen, m, it, st, par in SOFT_CASES:
        b, s = soft_inputs(n, gen)
        im = "box" if tag.endswith("_box") else "rbox"
        keep = middle(b, s, iou_method=im, iou_threshold=it, score_threshold=st, supression_method=m, supression_param=par)
        exp = np.unpackbits(g[tag])[:n].astype(bool)
        assert np.array_equal(keep, exp), (tag, int((keep != exp).sum()))


def test_small_frames_vs_oracle(dev, oracle):
    from d3d_b200.box import box2d_nms_batch
    rng = np.random.default_rng(77)
    frames = [(gen_boxes(rng, n, spread=4.0), rng.random(n)) for n in (1, 2, 65, 300)]
    for im in ("box", "rbox"):
        for m, par in (("linear", 0.7), ("gaussian", 0.4)):
            keeps = box2d_nms_batch([b for b, _ in frames], [s for _, s in frames], iou_method=im, iou_threshold=0.2, score_threshold=0.25,
                                    supression_method=m, supression_param=par)   # numpy in, numpy out
            for (b, s), k in zip(frames, keeps):
                assert isinstance(k, np.ndarray) and k.dtype == bool
                assert np.array_equal(k, oracle.box2d_nms(b, s, im, m, 0.2, 0.25, par, cuda_score_rule=True)), (im, m, len(b))


def test_crowd_frame_and_fallback_frame(dev):
    """a crowd of 2500 near-identical boxes has 3.1 M candidate pairs, far over the list capacity (32 x max_frame_boxes): the frame
    decays over all boxes behind the kept one; a frame of 9000 boxes takes one box2d_nms call per frame"""
    from d3d_b200.box import box2d_nms
    rng = np.random.default_rng(3)
    crowd = (np.array([5.0, 5.0, 4.0, 2.0, 0.3]) + rng.normal(0, 0.02, (2500, 5)), rng.random(2500))
    for frames in ([crowd] + _frames(rng, (500,)), _frames(rng, (9000, 100))):
        for im in ("box", "rbox"):
            for m in ("linear", "gaussian"):
                _check_per_frame(dev, frames, im, m, 0.3, 0.1, True, np.float64)
    b, s = crowd
    keep = box2d_nms(b, s, "rbox", "gaussian", iou_threshold=0.3, score_threshold=0.1, supression_param=0.5)
    assert 0 < keep.sum() < 2500


def test_call_forms(dev):
    from d3d_b200.box import box2d_nms_batch
    rng = np.random.default_rng(21)
    frames = _frames(rng, (400, 0, 90))
    kw = dict(iou_method="rbox", iou_threshold=0.3, score_threshold=0.2, supression_method="gaussian", supression_param=0.5)
    lst = box2d_nms_batch([_t(b, dev) for b, _ in frames], [_t(s, dev) for _, s in frames], **kw)
    off = np.cumsum([0] + [len(b) for b, _ in frames])
    pb, ps = np.concatenate([b for b, _ in frames]), np.concatenate([s for _, s in frames])
    packed = box2d_nms_batch(_t(pb, dev), _t(ps, dev), torch.from_numpy(off), offsets_dev=torch.from_numpy(off).to(dev), **kw)
    assert packed.is_cuda and torch.equal(packed, torch.cat(lst))
    packed_np = box2d_nms_batch(pb, ps, off, **kw)   # numpy in, numpy out
    assert isinstance(packed_np, np.ndarray) and np.array_equal(packed_np, packed.cpu().numpy())
    packed32 = box2d_nms_batch(_t(pb.astype(np.float32), dev), _t(ps.astype(np.float32), dev), torch.from_numpy(off), precise=False, **kw)
    lst32 = box2d_nms_batch([_t(b.astype(np.float32), dev) for b, _ in frames], [_t(s.astype(np.float32), dev) for _, s in frames],
                            precise=False, **kw)
    assert torch.equal(packed32, torch.cat(lst32))
    assert box2d_nms_batch([], [], supression_method="linear") == []
    hard = box2d_nms_batch(_t(pb, dev), _t(ps, dev), torch.from_numpy(off), iou_method="rbox", iou_threshold=0.3, score_threshold=0.2)
    assert torch.equal(hard, box2d_nms_batch(_t(pb, dev), _t(ps, dev), torch.from_numpy(off), iou_method="rbox", iou_threshold=0.3,
                                             score_threshold=0.2, supression_method="hard"))


def test_cabi_arguments(dev):
    b = torch.zeros((10, 5), dtype=torch.float64, device=dev)
    s = torch.ones(10, dtype=torch.float64, device=dev)
    off = torch.tensor([0, 4, 10], dtype=torch.int64, device=dev)
    sup = torch.zeros(10, dtype=torch.uint8, device=dev)
    need = _cabi.nms_batch_soft_workspace_bytes(10, 2, 6, _cabi.F64)
    ws = torch.empty(need, dtype=torch.uint8, device=dev)

    def call(sup_type, nbytes=need, mfb=6):
        return _cabi.nms2d_batch_soft[_cabi.F64](_cabi.ptr(b), _cabi.ptr(s), 10, _cabi.ptr(off), 2, mfb, 1, sup_type, 0.3, 0.1, 0.5,
                                                 _cabi.ptr(sup), _cabi.ptr(ws), nbytes, _cabi.stream_ptr())

    assert call(1) == _cabi.OK and call(2) == _cabi.OK
    assert call(0) == _cabi.ERR_INVALID   # hard NMS has its own entry point
    assert call(3) == _cabi.ERR_INVALID and call(-1) == _cabi.ERR_INVALID
    assert call(1, nbytes=need - 1) == _cabi.ERR_WORKSPACE
    big = _cabi.nms_batch_soft_workspace_bytes(9000, 1, 9000, _cabi.F64)
    assert _cabi.nms2d_batch_soft[_cabi.F64](_cabi.ptr(b), _cabi.ptr(s), 9000, _cabi.ptr(off), 1, 9000, 1, 1, 0.3, 0.1, 0.5, _cabi.ptr(sup),
                                            _cabi.ptr(ws), big, _cabi.stream_ptr()) == _cabi.ERR_UNSUPPORTED
    hard_ws = torch.empty(_cabi.nms_batch_workspace_bytes(10, 2, 6, _cabi.F64), dtype=torch.uint8, device=dev)
    assert _cabi.nms2d_batch[_cabi.F64](_cabi.ptr(b), _cabi.ptr(s), 10, _cabi.ptr(off), 2, 6, 1, 1, 0.3, 0.1, _cabi.ptr(sup), _cabi.ptr(hard_ws),
                                        hard_ws.numel(), _cabi.stream_ptr()) == _cabi.ERR_UNSUPPORTED
    torch.cuda.synchronize()
