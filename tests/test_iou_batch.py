"""Frame-batched differentiable IoU family (box2d_iou_batch over d3d_box2d_iou_batch_* / d3d_box2d_iou_batch_backward_*): per frame the
values and both gradients equal box2d_iou on that frame bit for bit, for every method, precision and call form; small frames agree with the
local-frame float64 reference; launch counts do not grow with the number of frames."""
import ctypes as C

import numpy as np
import pytest
import torch

import iou_ex_cases as IC
from conftest import gen_boxes, golden
from d3d_b200 import _cabi

METHODS = pytest.mark.parametrize("method", ["box", "rbox", "grbox", "drbox"])
DTS = pytest.mark.parametrize("dt", [np.float32, np.float64], ids=["f32", "f64"])
SIDES = (0, 1, 7, 63, 64, 65, 127, 128, 129, 257)


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda:0")


def _t(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def _bits(x):
    a = np.ascontiguousarray(x.detach().cpu().numpy() if torch.is_tensor(x) else x)
    return a.view(np.uint32 if a.dtype == np.float32 else np.uint64)


def _boxes(rng, n, dt, shift=0.0, scale=(1, 1, 1, 1, 1)):
    b = gen_boxes(rng, n) * scale
    b[:, :2] += shift
    return b.astype(dt)


# ------------------------------------------------------------------ C ABI, no GPU needed
def test_cabi_return_codes_without_gpu():
    """argument errors return codes before any CUDA call; empty batches are a no-op"""
    lib = C.CDLL(_cabi.LIB_PATH)
    i64, vp, sz = C.c_int64, C.c_void_p, C.c_size_t
    wsb = lib.d3d_box2d_iou_batch_workspace_bytes
    wsb.restype, wsb.argtypes = sz, [i64, i64, i64, C.c_int]
    need = wsb(20, 30, 3, 0)
    assert need >= (20 + 3 * 64) * 32 + (30 + 3 * 128) * 32 and wsb(20, 30, 3, 1) >= (20 + 3 * 64 + 30 + 3 * 64) * 64
    assert wsb(-1, 30, 3, 0) == 0 and wsb(20, 30, -1, 1) == 0
    names = ["b1", "t1", "o1", "b2", "t2", "o2", "nf", "mx1", "mx2", "type", "oo"]
    ok = [8, 20, 8, 8, 30, 8, 3, 10, 16, 2, 8]
    calls = {}
    for s in ("f32", "f64"):
        fw, bw = getattr(lib, f"d3d_box2d_iou_batch_{s}"), getattr(lib, f"d3d_box2d_iou_batch_backward_{s}")
        fw.argtypes = [vp, i64, vp, vp, i64, vp, i64, i64, i64, C.c_int, vp, vp, vp, sz, vp]
        bw.argtypes = [vp, i64, vp, vp, i64, vp, i64, i64, i64, C.c_int, vp, vp, vp, vp, vp]
        calls[f"fwd_{s}"] = (fw, names + ["out", "ws", "wsb", "st"], ok + [8, 8, wsb(20, 30, 3, 0 if s == "f32" else 1), 0])
        calls[f"bwd_{s}"] = (bw, names + ["grad", "g1", "g2", "st"], ok + [8, 8, 8, 0])
    for what, (fn, keys, base) in calls.items():
        def call(**kw):
            a = list(base)
            for k, v in kw.items():
                a[keys.index(k)] = v
            return fn(*a)
        for k in ("t1", "t2", "nf", "mx1", "mx2"):
            assert call(**{k: -1}) == _cabi.ERR_INVALID, (what, k)
        for t in (0, 3, 5, 7, -1):
            assert call(type=t) == _cabi.ERR_INVALID and call(type=t, nf=0) == _cabi.ERR_INVALID, (what, t)
        for t in (1, 2, 4, 6):
            assert call(type=t, nf=0) == _cabi.OK, (what, t)
        assert call(nf=0, b1=0, b2=0, o1=0, o2=0, oo=0) == _cabi.OK, what
        for k in ("o1", "o2", "oo", "b1", "b2"):
            assert call(**{k: 0}) == _cabi.ERR_INVALID, (what, k)
        if what.startswith("fwd"):
            assert call(t1=0) == _cabi.OK and call(t2=0) == _cabi.OK, what
            for t in (1, 2):   # "box" / "rbox" need the workspace; "grbox" / "drbox" need none
                assert call(type=t, wsb=base[-2] - 1) == _cabi.ERR_WORKSPACE and call(type=t, ws=0) == _cabi.ERR_WORKSPACE, (what, t)
            assert call(type=2, mx1=65535 * 64 + 1) == _cabi.ERR_UNSUPPORTED, what
            assert call(out=0) == _cabi.ERR_INVALID, what
        else:
            assert call(grad=0) == _cabi.ERR_INVALID and call(g1=0) == _cabi.ERR_INVALID and call(g2=0) == _cabi.ERR_INVALID, what


# ------------------------------------------------------------------ values
def _single(a, b, method, precise):
    from d3d_b200.box import box2d_iou
    return box2d_iou(a, b, method, precise)


def _value_frames(rng, dt):
    """ragged frames of the SIDES sizes, a frame 1 km (fp32) or 100 km (fp64) from the origin, the iou_degenerate.npz pairs, a NaN box"""
    frames = [(_boxes(rng, n, dt), _boxes(rng, m, dt)) for n, m in
              [(0, 7), (7, 0), (0, 0), (1, 1), (1, 64), (7, 63), (63, 65), (64, 64), (65, 127), (127, 128), (128, 129), (129, 257), (257, 7),
               (257, 129), (65, 1)]]
    far = 1e3 if dt == np.float32 else 1e5
    frames.insert(5, (_boxes(rng, 40, dt, far), _boxes(rng, 70, dt, far)))
    g = golden("iou_degenerate.npz")
    frames.insert(9, (g["boxes1"].astype(dt), g["boxes2"].astype(dt)))
    a, b = _boxes(rng, 9, dt), _boxes(rng, 11, dt)
    a[2, 0], b[4, 4] = np.nan, np.nan
    frames.append((a, b))
    return frames


@pytest.mark.gpu
@METHODS
@DTS
@pytest.mark.parametrize("precise", [True, False], ids=["precise", "native"])
def test_values_bit_equal_per_frame(dev, method, dt, precise):
    from d3d_b200.box import box2d_iou_batch
    rng = np.random.default_rng(3)
    frames = _value_frames(rng, dt)
    blocks = box2d_iou_batch([_t(a, dev) for a, _ in frames], [_t(b, dev) for _, b in frames], method=method, precise=precise)
    assert len(blocks) == len(frames)
    for f, (a, b) in enumerate(frames):
        v = _single(_t(a, dev), _t(b, dev), method, precise)
        assert blocks[f].dtype == v.dtype and tuple(blocks[f].shape) == (len(a), len(b)), f
        assert np.array_equal(_bits(blocks[f]), _bits(v)), (method, f, len(a), len(b))
    assert blocks[5].abs().sum() > 0


@pytest.mark.gpu
@METHODS
@pytest.mark.parametrize("dt,precise", [(np.float32, False), (np.float64, True)], ids=["f32", "f64"])
def test_tall_frame(dev, method, dt, precise):
    """a frame of 65 537 rows x 3 between small frames: more row tiles / owned-box warps than one grid.y slab of 65 535 rows; values and
    gradients"""
    from d3d_b200.box import box2d_iou_batch
    rng = np.random.default_rng(5)
    frames = [(_boxes(rng, 5, dt), _boxes(rng, 9, dt)), (_boxes(rng, 65537, dt, scale=(1, 1, .2, .2, 1)), _boxes(rng, 3, dt)),
              (_boxes(rng, 2, dt), _boxes(rng, 65537, dt))]
    l1, l2 = [_t(a, dev).requires_grad_(True) for a, _ in frames], [_t(b, dev).requires_grad_(True) for _, b in frames]
    blocks = box2d_iou_batch(l1, l2, method=method, precise=precise)
    sum(x.sum() for x in blocks).backward()
    for f, (a, b) in enumerate(frames):
        sa, sb = _t(a, dev).requires_grad_(True), _t(b, dev).requires_grad_(True)
        v = _single(sa, sb, method, precise)
        v.sum().backward()
        assert np.array_equal(_bits(blocks[f]), _bits(v)), (method, f)
        assert np.array_equal(_bits(l1[f].grad), _bits(sa.grad)) and np.array_equal(_bits(l2[f].grad), _bits(sb.grad)), (method, f)
    assert (blocks[1] != 0).any()


# ------------------------------------------------------------------ gradients
@pytest.mark.gpu
@METHODS
@pytest.mark.parametrize("dt,precise", [(np.float32, False), (np.float64, False), (np.float32, True)], ids=["f32", "f64", "f32-precise"])
def test_gradients_bit_equal_per_frame(dev, method, dt, precise):
    """packed form, a non-contiguous upstream gradient with ~90 % exact zeros; frames with an empty side get exact zeros"""
    from d3d_b200.box import box2d_iou_batch
    rng = np.random.default_rng(7)
    sizes = [(0, 5), (6, 0), (1, 1), (7, 63), (64, 65), (129, 33), (33, 257), (40, 40)]
    frames = [(_boxes(rng, n, dt), _boxes(rng, m, dt)) for n, m in sizes]
    frames.insert(4, (_boxes(rng, 30, dt, 1e3), _boxes(rng, 20, dt, 1e3)))
    o1, o2 = np.cumsum([0] + [len(a) for a, _ in frames]), np.cumsum([0] + [len(b) for _, b in frames])
    A = _t(np.concatenate([a for a, _ in frames]), dev).requires_grad_(True)
    B = _t(np.concatenate([b for _, b in frames]), dev).requires_grad_(True)
    flat, off = box2d_iou_batch(A, B, o1, o2, method=method, precise=precise)
    up = rng.normal(size=2 * flat.numel()) * (rng.random(2 * flat.numel()) < 0.1)
    upt = _t(up.astype(dt), dev)[::2]
    assert not upt.is_contiguous()
    flat.backward(upt)
    for f, (a, b) in enumerate(frames):
        sa, sb = _t(a, dev).requires_grad_(True), _t(b, dev).requires_grad_(True)
        v = _single(sa, sb, method, precise)
        v.backward(upt[int(off[f]):int(off[f + 1])].reshape(v.shape))
        ga, gb = A.grad[o1[f]:o1[f + 1]], B.grad[o2[f]:o2[f + 1]]
        sga = sa.grad if sa.grad is not None else torch.zeros_like(sa)
        sgb = sb.grad if sb.grad is not None else torch.zeros_like(sb)
        assert np.array_equal(_bits(ga), _bits(sga)) and np.array_equal(_bits(gb), _bits(sgb)), (method, f)
        if len(a) == 0 or len(b) == 0:
            assert not _bits(ga).any() and not _bits(gb).any(), f   # exact +0
    assert A.grad.abs().sum() > 0 and B.grad.abs().sum() > 0


@pytest.mark.gpu
@METHODS
@DTS
def test_vs_local_reference(dev, oracle, method, dt):
    """small frames against the local-frame float64 reference (oracle.iou_ex_local / iou_ex_grad_local) within iou_ex_cases.TOL, one of
    them moved far from the origin; each case frame is packed between two others"""
    from d3d_b200.box import box2d_iou_batch
    rng = np.random.default_rng(11)
    vt, gt = IC.TOL[dt]
    for off in (0.0, IC.OFFSETS[dt][-1]):
        a, b = IC.shifted(gen_boxes(rng, 6) + [0, 0, .3, .3, 0], gen_boxes(rng, 9) + [0, 0, .3, .3, 0], off, rng)
        a, b = a.astype(dt), b.astype(dt)
        up = rng.normal(size=(6, 9)).astype(dt)
        v, g1, g2, upm, smooth = IC.reference(oracle, a, b, method, up)
        assert smooth.mean() > 0.7
        frames = [(_boxes(rng, 4, dt), _boxes(rng, 3, dt)), (a, b), (_boxes(rng, 2, dt), _boxes(rng, 5, dt))]
        l1, l2 = [_t(x, dev).requires_grad_(True) for x, _ in frames], [_t(x, dev).requires_grad_(True) for _, x in frames]
        blocks = box2d_iou_batch(l1, l2, method=method, precise=False)
        (blocks[1] * _t(upm, dev)).sum().backward()
        # the "box" forward takes the AABB extents in absolute fp32 coordinates, as box2d_iou does: 2.2e-5 at 1 km
        assert IC.rel_err(blocks[1].detach().cpu().numpy(), v) <= (1e-4 if (method == "box" and dt == np.float32 and off >= 1e3) else vt), (method, off)
        assert IC.rel_err(l1[1].grad.cpu().numpy(), g1) <= gt and IC.rel_err(l2[1].grad.cpu().numpy(), g2) <= gt, (method, off)
        assert l1[0].grad is None or not l1[0].grad.any()


# ------------------------------------------------------------------ frame count, launches
@pytest.mark.gpu
@pytest.mark.parametrize("method,dt", [("rbox", np.float32), ("box", np.float64), ("grbox", np.float64), ("drbox", np.float32)])
def test_over_65535_frames(dev, method, dt):
    """70 000 frames of 1-8 boxes a side, packed: frames on grid.x beyond 65 535; a sample of frames against box2d_iou, values and gradients"""
    from d3d_b200.box import box2d_iou_batch
    rng = np.random.default_rng(13)
    nf = 70000
    ns, ms = rng.integers(1, 9, nf), rng.integers(1, 9, nf)
    A, B = _boxes(rng, int(ns.sum()), dt, scale=(.3, .3, 1, 1, 1)), _boxes(rng, int(ms.sum()), dt, scale=(.3, .3, 1, 1, 1))
    o1, o2 = np.cumsum(np.r_[0, ns]), np.cumsum(np.r_[0, ms])
    At, Bt = _t(A, dev).requires_grad_(True), _t(B, dev).requires_grad_(True)
    flat, off = box2d_iou_batch(At, Bt, o1, o2, method=method, precise=False)
    assert off.tolist() == np.cumsum(np.r_[0, ns * ms]).tolist()
    flat.sum().backward()
    for f in list(range(0, nf, 499)) + list(range(65530, 65541)) + list(range(nf - 20, nf)):
        sa, sb = _t(A[o1[f]:o1[f + 1]], dev).requires_grad_(True), _t(B[o2[f]:o2[f + 1]], dev).requires_grad_(True)
        v = _single(sa, sb, method, False)
        v.sum().backward()
        assert np.array_equal(_bits(flat[int(off[f]):int(off[f + 1])]), _bits(v.reshape(-1))), f
        assert np.array_equal(_bits(At.grad[o1[f]:o1[f + 1]]), _bits(sa.grad)) and np.array_equal(_bits(Bt.grad[o2[f]:o2[f + 1]]), _bits(sb.grad)), f
    assert (flat > 0).float().mean() > 0.05


@pytest.mark.gpu
@METHODS
def test_launch_count_independent_of_frames(dev, method):
    from d3d_b200.box import box2d_iou_batch
    rng = np.random.default_rng(17)

    def launches(nf):
        l1 = [_t(_boxes(rng, int(rng.integers(1, 50)), np.float32), dev).requires_grad_(True) for _ in range(nf)]
        l2 = [_t(_boxes(rng, int(rng.integers(1, 50)), np.float32), dev).requires_grad_(True) for _ in range(nf)]
        c0 = _cabi.launch_count()
        out = box2d_iou_batch(l1, l2, method=method, precise=False)
        c1 = _cabi.launch_count()
        sum(x.sum() for x in out).backward()
        return c1 - c0, _cabi.launch_count() - c1
    few, many = launches(2), launches(300)
    assert few == many, (few, many)
    assert few == ((1, 2) if method in ("grbox", "drbox") else (3, 2))


# ------------------------------------------------------------------ call forms
@pytest.mark.gpu
@METHODS
def test_call_forms(dev, method):
    """list and packed forms agree; numpy in -> numpy out; host tensors in -> host tensors out; list-form gradients reach every per-frame
    leaf; the argument errors of box2d_iou"""
    from d3d_b200.box import box2d_iou_batch
    rng = np.random.default_rng(19)
    sizes = [(40, 7), (0, 3), (17, 9), (5, 0), (300, 11)]
    fr = [(_boxes(rng, n, np.float64), _boxes(rng, m, np.float64)) for n, m in sizes]
    o1, o2 = np.cumsum([0] + [n for n, _ in sizes]), np.cumsum([0] + [m for _, m in sizes])
    A, Bx = np.concatenate([a for a, _ in fr]), np.concatenate([b for _, b in fr])
    kw = dict(method=method)

    lst = box2d_iou_batch([_t(a, dev) for a, _ in fr], [_t(b, dev) for _, b in fr], **kw)
    flat, off = box2d_iou_batch(_t(A, dev), _t(Bx, dev), torch.from_numpy(o1), torch.from_numpy(o2), **kw)
    assert flat.is_cuda and off.device.type == "cpu" and off.tolist() == np.cumsum([0] + [n * m for n, m in sizes]).tolist()
    assert np.array_equal(_bits(flat), _bits(torch.cat([x.reshape(-1) for x in lst])))
    assert all(x.untyped_storage().data_ptr() == lst[0].untyped_storage().data_ptr() for x in lst)   # views into one buffer
    assert all(tuple(x.shape) == s for x, s in zip(lst, sizes))
    flat_np, off_np = box2d_iou_batch(A, Bx, o1, o2, **kw)
    assert isinstance(flat_np, np.ndarray) and isinstance(off_np, np.ndarray) and np.array_equal(_bits(flat_np), _bits(flat))
    lst_np = box2d_iou_batch([a for a, _ in fr], [b for _, b in fr], **kw)
    assert all(isinstance(x, np.ndarray) and x.shape == s for x, s in zip(lst_np, sizes))
    flat_cpu, _ = box2d_iou_batch(torch.from_numpy(A), torch.from_numpy(Bx), o1, o2, **kw)
    assert flat_cpu.device.type == "cpu" and np.array_equal(_bits(flat_cpu), _bits(flat))
    lst_cpu = box2d_iou_batch([torch.from_numpy(a) for a, _ in fr], [torch.from_numpy(b) for _, b in fr], **kw)
    assert all(x.device.type == "cpu" for x in lst_cpu)
    f32, _ = box2d_iou_batch(_t(A, dev).float(), _t(Bx, dev).float(), o1, o2, precise=True, **kw)
    assert f32.dtype == torch.float32
    # non-contiguous: every other row of a doubled array, and a transposed copy
    A2, B2 = _t(np.repeat(A, 2, 0), dev)[::2], _t(np.ascontiguousarray(Bx.T), dev).t()
    assert not A2.is_contiguous() and not B2.is_contiguous()
    assert np.array_equal(_bits(box2d_iou_batch(A2, B2, o1, o2, **kw)[0]), _bits(flat))
    assert box2d_iou_batch([], [], **kw) == []
    f0, z0 = box2d_iou_batch(torch.zeros((0, 5), dtype=torch.float64), torch.zeros((0, 5), dtype=torch.float64), [0], [0], **kw)
    assert f0.numel() == 0 and z0.tolist() == [0]
    # list-form autograd reaches every per-frame leaf, host leaves included
    for d in (dev, torch.device("cpu")):
        l1, l2 = [torch.from_numpy(a).to(d).requires_grad_(True) for a, _ in fr], [torch.from_numpy(b).to(d).requires_grad_(True) for _, b in fr]
        sum(x.sum() for x in box2d_iou_batch(l1, l2, **kw)).backward()
        for (a, b), g1, g2 in zip(fr, l1, l2):
            assert g1.grad is not None and g2.grad is not None and g1.grad.device == d and g1.grad.shape == g1.shape
            sa, sb = _t(a, dev).requires_grad_(True), _t(b, dev).requires_grad_(True)
            _single(sa, sb, method, True).sum().backward()
            assert np.array_equal(_bits(g1.grad), _bits(sa.grad)) and np.array_equal(_bits(g2.grad), _bits(sb.grad))
    # the errors of box2d_iou
    with pytest.raises(ValueError, match="Nx2"):
        box2d_iou_batch([np.zeros((4, 5, 1))], [np.zeros((2, 5))], **kw)
    with pytest.raises(ValueError, match="fields"):
        box2d_iou_batch([np.zeros((4, 5))], [np.zeros((2, 4))], **kw)
    with pytest.raises(ValueError, match="fields"):
        box2d_iou_batch(A[:, :4], Bx, o1, o2, **kw)
    with pytest.raises(ValueError, match="Unrecognized iou type"):
        box2d_iou_batch(A, Bx, o1, o2, method="gbox")
    with pytest.raises(RuntimeError):
        box2d_iou_batch([_t(A, dev).float()], [_t(Bx, dev)], method=method, precise=False)
    with pytest.raises(ValueError):   # frame counts / offsets inconsistent
        box2d_iou_batch(A, Bx, o1[:-1], o2, **kw)
    with pytest.raises(ValueError):
        box2d_iou_batch(A, Bx, o1, o2 + 1, **kw)
    with pytest.raises(ValueError):
        box2d_iou_batch(A, Bx, **kw)
    with pytest.raises(ValueError):
        box2d_iou_batch([A], [Bx, Bx], **kw)
    torch.cuda.synchronize()


@pytest.mark.gpu
def test_rbox_frame_past_tile_grid(dev):
    """an fp64 "rbox" frame of 65 535 * 64 + 1 rows (one row tile more than grid.z holds) takes the single-frame kernel into its block;
    the frames around it take the batch kernel, and values and gradients match box2d_iou"""
    from d3d_b200.box import box2d_iou_batch
    rng = np.random.default_rng(23)
    big = _boxes(rng, 65535 * 64 + 1, np.float64, scale=(1, 1, .2, .2, 1))
    frames = [(_boxes(rng, 30, np.float64), _boxes(rng, 20, np.float64)), (big, _boxes(rng, 2, np.float64)),
              (_boxes(rng, 9, np.float64), _boxes(rng, 70, np.float64))]
    c0 = _cabi.launch_count()
    l1, l2 = [_t(a, dev).requires_grad_(True) for a, _ in frames], [_t(b, dev).requires_grad_(True) for _, b in frames]
    blocks = box2d_iou_batch(l1, l2, method="rbox")
    assert _cabi.launch_count() - c0 == 3 + 3   # the batch (2 preps + tiles) and the single frame (2 preps + tiles)
    sum(x.sum() for x in blocks).backward()
    for f, (a, b) in enumerate(frames):
        sa, sb = _t(a, dev).requires_grad_(True), _t(b, dev).requires_grad_(True)
        v = _single(sa, sb, "rbox", True)
        v.sum().backward()
        assert np.array_equal(_bits(blocks[f]), _bits(v)), f
        assert np.array_equal(_bits(l1[f].grad), _bits(sa.grad)) and np.array_equal(_bits(l2[f].grad), _bits(sb.grad)), f
    assert (blocks[1] > 0).any()
