"""Fused max-IoU reduction (box2d_iou_max / box2d_iou_max_batch over d3d_box2d_iou_max_batch_*): per frame the four outputs equal
torch.max(box2d_iou(...), dim=1 / dim=0) on that frame bit for bit (NaN matches NaN), for "box" and "rbox", fp32 and fp64, precise on and
off; a box whose frame's other side is empty gets (0, -1)."""
import ctypes as C

import numpy as np
import pytest
import torch

from conftest import gen_boxes, golden
from d3d_b200 import _cabi

METHODS = pytest.mark.parametrize("method", ["box", "rbox"])
DTS = pytest.mark.parametrize("dt", [np.float32, np.float64], ids=["f32", "f64"])
PRECISE = pytest.mark.parametrize("precise", [True, False], ids=["precise", "native"])


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda:0")


def _t(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def _boxes(rng, n, dt, shift=0.0, scale=(1, 1, 1, 1, 1)):
    b = gen_boxes(rng, n) * scale
    b[:, :2] += shift
    return b.astype(dt)


def _same(x, y):
    """same dtype and shape, NaN where the other is NaN, every other element bit-equal"""
    x, y = torch.as_tensor(x).cpu(), torch.as_tensor(y).cpu()
    if x.dtype != y.dtype or x.shape != y.shape:
        return False
    if x.is_floating_point():
        nx, ny = torch.isnan(x), torch.isnan(y)
        iv = torch.int32 if x.dtype == torch.float32 else torch.int64
        return bool(torch.equal(nx, ny) and torch.equal(x.view(iv)[~nx], y.view(iv)[~ny]))
    return bool(torch.equal(x, y))


def _reference(a, b, method, precise):
    """torch.max of box2d_iou's matrix along both axes; (0, -1) where the other side is empty"""
    from d3d_b200.box import box2d_iou
    v = box2d_iou(a, b, method, precise)
    n, m = v.shape
    if n and m:
        (m1, i1), (m2, i2) = v.max(1), v.max(0)
    else:
        m1, i1 = torch.zeros(n, dtype=v.dtype, device=v.device), torch.full((n,), -1, dtype=torch.int64, device=v.device)
        m2, i2 = torch.zeros(m, dtype=v.dtype, device=v.device), torch.full((m,), -1, dtype=torch.int64, device=v.device)
    return (m1, i1, m2, i2), v


def _check_frame(got, a, b, method, precise, what):
    ref, v = _reference(a, b, method, precise)
    for k, (g, r) in enumerate(zip(got, ref)):
        assert _same(g, r), (what, k, tuple(a.shape), tuple(b.shape))
    return v


# ------------------------------------------------------------------ C ABI and front door, no GPU needed
def test_cabi_return_codes_without_gpu():
    """argument errors return codes before any CUDA call; an empty batch is a no-op"""
    lib = C.CDLL(_cabi.LIB_PATH)
    i64, vp, sz = C.c_int64, C.c_void_p, C.c_size_t
    wsb = lib.d3d_box2d_iou_max_batch_workspace_bytes
    wsb.restype, wsb.argtypes = sz, [i64, i64, i64, C.c_int]
    need32, need64 = wsb(20, 30, 3, 0), wsb(20, 30, 3, 1)
    assert need32 >= (20 + 3 * 64 + 30 + 3 * 128) * 32 + 50 * 8 and need64 >= (20 + 3 * 64 + 30 + 3 * 64) * 64 + 50 * 16
    assert wsb(-1, 30, 3, 0) == 0 and wsb(20, -1, 3, 1) == 0 and wsb(20, 30, -1, 0) == 0
    keys = ["b1", "t1", "o1", "b2", "t2", "o2", "nf", "mx1", "mx2", "type", "odt", "max1", "idx1", "max2", "idx2", "ws", "wsb", "st"]
    for s, code, need in (("f32", 0, need32), ("f64", 1, need64)):
        fn = getattr(lib, f"d3d_box2d_iou_max_batch_{s}")
        fn.argtypes = [vp, i64, vp, vp, i64, vp, i64, i64, i64, C.c_int, C.c_int, vp, vp, vp, vp, vp, sz, vp]
        base = [8, 20, 8, 8, 30, 8, 3, 10, 16, 2, code, 8, 8, 8, 8, 8, need, 0]

        def call(**kw):
            a = list(base)
            for k, v in kw.items():
                a[keys.index(k)] = v
            return fn(*a)
        for t in (0, 3, 4, 5, 6, 7, -1):   # "box" and "rbox" only
            assert call(type=t) == _cabi.ERR_INVALID and call(type=t, nf=0) == _cabi.ERR_INVALID, (s, t)
        for odt in (-1, 2) + ((1,) if s == "f32" else ()):   # fp64 outputs need fp64 boxes
            assert call(odt=odt) == _cabi.ERR_INVALID, (s, odt)
        for k in ("t1", "t2", "nf", "mx1", "mx2"):
            assert call(**{k: -1}) == _cabi.ERR_INVALID, (s, k)
        for t in (1, 2):
            assert call(type=t, nf=0) == _cabi.OK and call(type=t, t1=0, t2=0) == _cabi.OK, (s, t)
            assert call(type=t, wsb=need - 1) == _cabi.ERR_WORKSPACE and call(type=t, ws=0) == _cabi.ERR_WORKSPACE, (s, t)
        assert call(nf=0, b1=0, b2=0, o1=0, o2=0, max1=0, idx1=0, max2=0, idx2=0) == _cabi.OK, s
        for k in ("o1", "o2", "b1", "b2", "max1", "idx1", "max2", "idx2"):
            assert call(**{k: 0}) == _cabi.ERR_INVALID, (s, k)
        assert call(nf=1 << 31) == _cabi.ERR_UNSUPPORTED, s
        assert call(odt=0, mx1=1 << 32) == _cabi.ERR_UNSUPPORTED and call(odt=0, mx2=1 << 32) == _cabi.ERR_UNSUPPORTED, s   # 32-bit index of the fp32 key


def test_front_door_errors_without_gpu():
    """the errors of box2d_iou_batch, and "Unsupported iou type!" for the GIoU / DIoU methods, raised before any device work"""
    from d3d_b200.box import box2d_iou_max, box2d_iou_max_batch
    rng = np.random.default_rng(1)
    A, B = gen_boxes(rng, 9), gen_boxes(rng, 7)
    o1, o2 = np.array([0, 4, 9]), np.array([0, 7, 7])
    for m in ("grbox", "drbox"):
        with pytest.raises(ValueError, match="Unsupported iou type!"):
            box2d_iou_max(A, B, m)
        with pytest.raises(ValueError, match="Unsupported iou type!"):
            box2d_iou_max_batch(A, B, o1, o2, method=m)
        with pytest.raises(ValueError, match="Unsupported iou type!"):
            box2d_iou_max_batch([A], [B], method=m)
    with pytest.raises(ValueError, match="Nx2"):
        box2d_iou_max(A[:, :, None], B)
    with pytest.raises(ValueError, match="fields"):
        box2d_iou_max(A, B[:, :4])
    with pytest.raises(ValueError, match="Nx2"):
        box2d_iou_max_batch([np.zeros((4, 5, 1))], [np.zeros((2, 5))])
    with pytest.raises(ValueError, match="fields"):
        box2d_iou_max_batch(A[:, :4], B, o1, o2)
    with pytest.raises(ValueError):   # frame counts / offsets inconsistent
        box2d_iou_max_batch(A, B, o1[:-1], o2)
    with pytest.raises(ValueError):
        box2d_iou_max_batch(A, B, o1, o2 + 1)
    with pytest.raises(ValueError, match="ascending"):
        box2d_iou_max_batch(A, B, np.array([0, 5, 4, 9]), np.array([0, 7, 7, 7]))
    with pytest.raises(ValueError):
        box2d_iou_max_batch(A, B)
    with pytest.raises(ValueError):
        box2d_iou_max_batch([A], [B, B])
    with pytest.raises(RuntimeError):
        box2d_iou_max_batch([A, A.astype(np.float32)], [B, B])
    assert box2d_iou_max_batch([], []) == []


# ------------------------------------------------------------------ values
def _near_ties(rng, dt):
    """200 m x 10 m boxes: boxes2 centred 0 .. 199 float32 ulps right of x = 1, boxes1 at x = 0 .. 1.11.  The float64 IoUs of a row all
    differ, and dozens of them round to its largest float32 value, so precise=True must take the lowest index among the float32 ties,
    not the float64 maximum"""
    b = np.zeros((200, 5))
    b[:, 0] = (np.float32(1.0) + np.arange(200, dtype=np.float32) * np.float32(2 ** -23))[rng.permutation(200)]
    b[:, 2:4] = 200, 10
    a = np.zeros((4, 5))
    a[:, 0] = np.arange(4) * 0.37
    a[:, 2:4] = 200, 10
    return a.astype(dt), b.astype(dt)


def _value_frames(rng, dt):
    fr = [(_boxes(rng, n, dt), _boxes(rng, m, dt)) for n, m in [(0, 7), (7, 0), (0, 0), (1, 1)]]
    for n, m in [(63, 127), (64, 128), (65, 129), (63, 63), (64, 64), (65, 65), (129, 3), (3, 257)]:   # tile edges of fp32 and fp64
        fr.append((_boxes(rng, n, dt), _boxes(rng, m, dt)))
    fr.append((_boxes(rng, 70, dt), _boxes(rng, 140, dt, 1000.0)))   # every pair rejected: all +0, index 0
    fr.append((np.tile(_boxes(rng, 3, dt), (25, 1)), np.tile(_boxes(rng, 5, dt), (30, 1))))   # exact ties across tiles
    fr.append(_near_ties(rng, dt))
    fr.append((_boxes(rng, 40, dt, 1e5), _boxes(rng, 70, dt, 1e5)))   # 100 km from the origin
    g = golden("iou_degenerate.npz")
    fr.append((g["boxes1"].astype(dt), g["boxes2"].astype(dt)))
    a, b = _boxes(rng, 12, dt), _boxes(rng, 11, dt)
    a[2, 0], b[4, 4], a[5, 2], b[7, 3], a[8, 1] = np.nan, np.nan, np.inf, np.inf, -np.inf
    a[9, 2:4], b[9, 2:4] = 0, 0          # zero-area boxes: "box" divides 0 / 0
    a[10, 2:4], b[10, 2:4] = 1e-20, 3e-20   # subnormal areas
    b[10, [0, 1, 4]] = a[10, [0, 1, 4]]   # same centre and heading: the pair is clipped
    fr.append((a, b))
    return fr


@pytest.mark.gpu
@METHODS
@DTS
@PRECISE
def test_values_bit_equal_per_frame(dev, method, dt, precise):
    """list form against torch.max of box2d_iou per frame; the matrices themselves hold no negative value and no -0 (so the initial key
    (+0, index 0) is the answer of a row without a positive value or NaN)"""
    from d3d_b200.box import box2d_iou_max_batch
    rng = np.random.default_rng(3)
    frames = _value_frames(rng, dt)
    out = box2d_iou_max_batch([_t(a, dev) for a, _ in frames], [_t(b, dev) for _, b in frames], method=method, precise=precise)
    assert len(out) == len(frames)
    nan_seen = False
    for f, (a, b) in enumerate(frames):
        assert all(not x.requires_grad for x in out[f])
        v = _check_frame(out[f], _t(a, dev), _t(b, dev), method, precise, (method, f))
        assert not bool((v < 0).any()) and not bool(((v == 0) & torch.signbit(v)).any()), (method, f)
        nan_seen |= bool(torch.isnan(v).any())
    assert nan_seen or method == "rbox"   # "box": NaN boxes and 0 / 0; "rbox" rejects NaN boxes (+0)
    rej = out[12]
    assert bool((rej[0] == 0).all()) and not bool(torch.signbit(rej[0]).any()) and bool((rej[1] == 0).all())
    assert out[0][2].tolist() == [0.0] * 7 and out[0][3].tolist() == [-1] * 7 and out[1][0].tolist() == [0.0] * 7 and out[1][1].tolist() == [-1] * 7
    if precise and dt == np.float32:   # the near ties are decided on the rounded values
        from d3d_b200.box import box2d_iou
        a, b = frames[14]
        full = box2d_iou(_t(a, dev), _t(b, dev), method, True)
        exact = box2d_iou(_t(a, dev).double(), _t(b, dev).double(), method, False)
        assert bool((exact.max(1).indices != full.max(1).indices).any())


@pytest.mark.gpu
@METHODS
def test_over_65535_frames(dev, method):
    """70 000 frames of 0-8 boxes a side, packed: frames on grid.x beyond 65 535; a sample of frames against the reference"""
    from d3d_b200.box import box2d_iou_max_batch
    rng = np.random.default_rng(13)
    nf = 70000
    ns, ms = rng.integers(0, 9, nf), rng.integers(0, 9, nf)
    A, B = _boxes(rng, int(ns.sum()), np.float32, scale=(.3, .3, 1, 1, 1)), _boxes(rng, int(ms.sum()), np.float32, scale=(.3, .3, 1, 1, 1))
    o1, o2 = np.cumsum(np.r_[0, ns]), np.cumsum(np.r_[0, ms])
    for precise in (False, True):
        m1, i1, m2, i2 = box2d_iou_max_batch(_t(A, dev), _t(B, dev), o1, o2, method=method, precise=precise)
        assert m1.shape == (len(A),) and m2.shape == (len(B),) and i1.dtype == torch.int64
        for f in list(range(0, nf, 499)) + list(range(65530, 65541)) + list(range(nf - 20, nf)):
            s1, s2 = slice(o1[f], o1[f + 1]), slice(o2[f], o2[f + 1])
            _check_frame((m1[s1], i1[s1], m2[s2], i2[s2]), _t(A[s1], dev), _t(B[s2], dev), method, precise, f)
        assert bool((m1 > 0).float().mean() > 0.3)


@pytest.mark.gpu
@METHODS
def test_frame_past_tile_grid(dev, method):
    """one frame of 65 535 * 64 + 65 rows x 3: more row tiles than one launch holds ("rbox": 64-row tiles, "box": 32-row chunks), so the
    C call launches the tiles in slabs and the keys combine across them"""
    from d3d_b200.box import box2d_iou_max
    rng = np.random.default_rng(23)
    a = _boxes(rng, 65535 * 64 + 65, np.float32, scale=(1, 1, .3, .3, 1))
    b = _boxes(rng, 3, np.float32)
    a[-3:] = b   # IoU 1 in the last slab
    c0 = _cabi.launch_count()
    got = box2d_iou_max(_t(a, dev), _t(b, dev), method, precise=False)
    assert _cabi.launch_count() - c0 == (4 + (2 if method == "rbox" else 3))   # init, 2 preps, tile slabs, finalise
    _check_frame(got, _t(a, dev), _t(b, dev), method, False, "tall")
    assert got[3].tolist() == list(range(len(a) - 3, len(a)))


@pytest.mark.gpu
@METHODS
@pytest.mark.parametrize("precise", [False, True], ids=["native", "precise"])
def test_c1_frame(dev, method, precise):
    """one 20 000 x 20 000 frame of the C1 distribution, fp32 boxes"""
    from d3d_b200.box import box2d_iou_max
    rng = np.random.default_rng(29)
    a, b = _t(gen_boxes(rng, 20000).astype(np.float32), dev), _t(gen_boxes(rng, 20000).astype(np.float32), dev)
    got = box2d_iou_max(a, b, method, precise)
    _check_frame(got, a, b, method, precise, "c1")
    torch.cuda.empty_cache()


# ------------------------------------------------------------------ call forms, determinism, launches
@pytest.mark.gpu
@METHODS
def test_call_forms(dev, method):
    """list and packed forms agree (packed indices are frame-local); numpy in -> numpy out; host tensors in -> host tensors out; the
    single-frame function equals a one-frame batch; repeated calls give identical outputs"""
    from d3d_b200.box import box2d_iou_max, box2d_iou_max_batch
    rng = np.random.default_rng(19)
    sizes = [(40, 7), (0, 3), (17, 9), (5, 0), (300, 11), (70, 300)]
    fr = [(_boxes(rng, n, np.float64), _boxes(rng, m, np.float64)) for n, m in sizes]
    o1, o2 = np.cumsum([0] + [n for n, _ in sizes]), np.cumsum([0] + [m for _, m in sizes])
    A, Bx = np.concatenate([a for a, _ in fr]), np.concatenate([b for _, b in fr])
    kw = dict(method=method)
    lst = box2d_iou_max_batch([_t(a, dev) for a, _ in fr], [_t(b, dev) for _, b in fr], **kw)
    packed = box2d_iou_max_batch(_t(A, dev), _t(Bx, dev), torch.from_numpy(o1), torch.from_numpy(o2), **kw)
    assert all(x.is_cuda for x in packed) and [x.dtype for x in packed] == [torch.float64, torch.int64] * 2
    for k in range(4):
        assert _same(packed[k], torch.cat([t[k] for t in lst]))
    for f, (a, b) in enumerate(fr):
        assert all(_same(x, y) for x, y in zip(lst[f], box2d_iou_max(_t(a, dev), _t(b, dev), method))), f
    for _ in range(3):
        assert all(_same(x, y) for x, y in zip(packed, box2d_iou_max_batch(_t(A, dev), _t(Bx, dev), o1, o2, **kw)))
    np_out = box2d_iou_max_batch(A, Bx, o1, o2, **kw)
    assert all(isinstance(x, np.ndarray) for x in np_out) and all(_same(torch.from_numpy(x), y) for x, y in zip(np_out, packed))
    lst_np = box2d_iou_max_batch([a for a, _ in fr], [b for _, b in fr], **kw)
    assert all(isinstance(x, np.ndarray) for t in lst_np for x in t) and all(len(t[0]) == n and len(t[2]) == m for t, (n, m) in zip(lst_np, sizes))
    host = box2d_iou_max_batch(torch.from_numpy(A), torch.from_numpy(Bx), o1, o2, **kw)
    assert all(x.device.type == "cpu" for x in host) and all(_same(x, y) for x, y in zip(host, packed))
    one_np = box2d_iou_max(fr[0][0], fr[0][1], method)
    assert all(isinstance(x, np.ndarray) for x in one_np) and all(_same(torch.from_numpy(x), y) for x, y in zip(one_np, lst[0]))
    f32 = box2d_iou_max_batch(_t(A, dev).float(), _t(Bx, dev).float(), o1, o2, precise=True, **kw)
    assert [x.dtype for x in f32] == [torch.float32, torch.int64] * 2
    g1 = _t(A, dev).requires_grad_(True)
    assert not any(x.requires_grad for x in box2d_iou_max_batch(g1, _t(Bx, dev), o1, o2, **kw))
    A2 = _t(np.repeat(A, 2, 0), dev)[::2]   # non-contiguous
    assert all(_same(x, y) for x, y in zip(box2d_iou_max_batch(A2, _t(Bx, dev), o1, o2, **kw), packed))
    z = box2d_iou_max_batch(torch.zeros((0, 5), dtype=torch.float64), torch.zeros((0, 5), dtype=torch.float64), [0], [0], **kw)
    assert all(x.numel() == 0 for x in z)
    e = box2d_iou_max(_t(A[:4], dev), _t(Bx[:0], dev), method)
    assert e[0].tolist() == [0.0] * 4 and e[1].tolist() == [-1] * 4 and e[2].numel() == 0
    torch.cuda.synchronize()


@pytest.mark.gpu
@METHODS
def test_launch_count_independent_of_frames(dev, method):
    from d3d_b200.box import box2d_iou_max_batch
    rng = np.random.default_rng(17)

    def launches(nf):
        l1 = [_t(_boxes(rng, int(rng.integers(1, 50)), np.float32), dev) for _ in range(nf)]
        l2 = [_t(_boxes(rng, int(rng.integers(1, 50)), np.float32), dev) for _ in range(nf)]
        c0 = _cabi.launch_count()
        box2d_iou_max_batch(l1, l2, method=method, precise=False)
        return _cabi.launch_count() - c0
    assert launches(2) == launches(300) == 5
