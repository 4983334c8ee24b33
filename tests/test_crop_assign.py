"""Fused reductions of the point-in-box mask (box2dr_crop_assign / box3dp_crop_assign and their batch forms over d3d_crop2dr_assign*):
per frame, point_box equals torch.where(mask.any(0), mask.to(torch.uint8).argmax(0), -1) and box_npoints equals mask.sum(1) exactly,
where mask is box2dr_crop / box3dp_crop on the same inputs, on the tile path and on the grid path."""
import ctypes as C

import numpy as np
import pytest
import torch

from conftest import gen_boxes, golden
from d3d_b200 import _cabi

DTS = pytest.mark.parametrize("dt", [np.float32, np.float64], ids=["f32", "f64"])
AXES = pytest.mark.parametrize("axis", [None, 0, 1, 2], ids=["2d", "ax0", "ax1", "ax2"])   # None: the 2-D functions
_PLANE = {0: ([1, 2], [1, 2, 4, 5, 6]), 1: ([0, 2], [0, 2, 3, 5, 6]), 2: ([0, 1], [0, 1, 3, 4, 6])}
PATHS = {"brute": 1, "grid": 2}


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda:0")


def _t(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def _frame(rng, n, m, axis, dt, shift=0.0):
    """n points around m boxes ([n, 2] / [m, 5], or [n, 3] / [m, 7] for a projection axis), moved by `shift` metres"""
    b2 = gen_boxes(rng, m) + [0, 0, .2, .2, 0]
    p2 = (rng.random((n, 2)) - .5) * 12
    if axis is None:
        b, p = b2, p2
    else:
        pc, bc = _PLANE[axis]
        b, p = np.zeros((m, 7)), np.zeros((n, 3))
        b[:, bc], p[:, pc] = b2, p2
        b[:, axis], b[:, 3 + axis] = rng.normal(0, 1, m), 0.5 + rng.random(m) * 3
        p[:, axis] = (rng.random(n) - .5) * 5
    p, b = p + shift, b.copy()
    b[:, :2 if axis is None else 3] += shift
    return p.astype(dt), b.astype(dt)


def _to3d(p2, b2, axis, pz=0.25, bz=0.5, bd=4.0):
    """3-D rows holding the 2-D frame in the plane of `axis`, every point inside the boxes' extent along it"""
    pc, bc = _PLANE[axis]
    p, b = np.zeros((len(p2), 3), p2.dtype), np.zeros((len(b2), 7), b2.dtype)
    p[:, pc], b[:, bc] = p2, b2
    p[:, axis], b[:, axis], b[:, 3 + axis] = pz, bz, bd
    return p, b


def _mask(p, b, axis):
    from d3d_b200.box import box2dr_crop, box3dp_crop
    return box2dr_crop(p, b) if axis is None else box3dp_crop(p, b, project_axis=axis)


def _reduce(mask):
    """the two reductions of a [M, N] mask"""
    mask = torch.as_tensor(mask)
    m, n = mask.shape
    if m == 0:
        return torch.full((n,), -1, dtype=torch.int64, device=mask.device), torch.zeros(0, dtype=torch.int64, device=mask.device)
    return torch.where(mask.any(0), mask.to(torch.uint8).argmax(0), -1), mask.sum(1)


def _assign(p, b, axis):
    from d3d_b200.box import box2dr_crop_assign, box3dp_crop_assign
    return box2dr_crop_assign(p, b) if axis is None else box3dp_crop_assign(p, b, project_axis=axis)


def _assign_batch(pl, bl, axis, **kw):
    from d3d_b200.box import box2dr_crop_assign_batch, box3dp_crop_assign_batch
    return box2dr_crop_assign_batch(pl, bl, **kw) if axis is None else box3dp_crop_assign_batch(pl, bl, project_axis=axis, **kw)


def _mask_batch(pl, bl, axis):
    from d3d_b200.box import box2dr_crop_batch, box3dp_crop_batch
    return box2dr_crop_batch(pl, bl) if axis is None else box3dp_crop_batch(pl, bl, project_axis=axis)


def _eq(got, ref, what):
    for g, r, name in zip(got, ref, ("point_box", "box_npoints")):
        g, r = torch.as_tensor(g).cpu(), torch.as_tensor(r).cpu()
        assert g.dtype == torch.int64 and g.shape == r.shape, (what, name, g.dtype, tuple(g.shape), tuple(r.shape))
        assert torch.equal(g, r), (what, name, int((g != r).sum()))


def _check_frames(frames, axis, dev, paths=(None,)):
    """batch (list form) and single-frame outputs against the reductions of the batch and single-frame masks"""
    pl, bl = [_t(p, dev) for p, _ in frames], [_t(b, dev) for _, b in frames]
    masks = _mask_batch(pl, bl, axis)
    refs = [_reduce(mk) for mk in masks]
    for path in paths:
        try:
            _cabi.tuning_set("D3D_B200_CROP_PATH", PATHS.get(path))
            got = _assign_batch(pl, bl, axis)
            assert len(got) == len(frames)
            for f, (p, b) in enumerate(zip(pl, bl)):
                _eq(got[f], refs[f], (path, axis, f, len(p), len(b), "batch"))
                _eq(_assign(p, b, axis), refs[f], (path, axis, f, len(p), len(b), "single"))
                _eq(_reduce(_mask(p, b, axis)), refs[f], (path, axis, f, "single mask"))
        finally:
            _cabi.tuning_set("D3D_B200_CROP_PATH", None)
    return refs


# ------------------------------------------------------------------ C ABI and front door, no GPU needed
def test_cabi_return_codes_without_gpu():
    """argument errors return codes before any CUDA call; an empty problem is a no-op"""
    lib = C.CDLL(_cabi.LIB_PATH)
    i64, vp, sz = C.c_int64, C.c_void_p, C.c_size_t
    wsb = lib.d3d_crop2dr_assign_batch_workspace_bytes
    wsb.restype, wsb.argtypes = sz, [i64, C.c_int]
    need = wsb(20, 0)
    assert need >= 20 * 48 and wsb(20, 1) >= 20 * 96 and wsb(-1, 0) == 0
    wss = lib.d3d_crop2dr_assign_workspace_bytes
    wss.restype, wss.argtypes = sz, [i64, i64, C.c_int]
    need1 = wss(30, 20, 0)
    assert need1 >= 30 * 16 + 20 * 48 and wss(30, 20, 1) > need1 and wss(-1, 20, 0) == 0 and wss(30, -1, 1) == 0

    names = ["p", "tp", "po", "b", "tb", "bo", "nf", "mxp", "mxb", "ax", "pb", "bn", "ws", "wsb", "st"]
    ok = [8, 30, 8, 8, 20, 8, 3, 16, 9, -1, 8, 8, 8, need, 0]
    snames = ["p", "n", "b", "m", "ax", "pb", "bn", "ws", "wsb", "st"]
    sok = [8, 30, 8, 20, -1, 8, 8, 8, need1, 0]
    for s in ("f32", "f64"):
        fb = getattr(lib, f"d3d_crop2dr_assign_batch_{s}")
        fb.argtypes = [vp, i64, vp, vp, i64, vp, i64, i64, i64, C.c_int, vp, vp, vp, sz, vp]
        fs = getattr(lib, f"d3d_crop2dr_assign_{s}")
        fs.argtypes = [vp, i64, vp, i64, C.c_int, vp, vp, vp, sz, vp]
        bw, sw = (need, need1) if s == "f32" else (wsb(20, 1), wss(30, 20, 1))
        call = lambda **kw: fb(*[kw.get(k, v) for k, v in zip(names, ok[:-2] + [bw, 0])])  # noqa: E731
        scall = lambda **kw: fs(*[kw.get(k, v) for k, v in zip(snames, sok[:-2] + [sw, 0])])  # noqa: E731
        for k in ("tp", "tb", "nf", "mxp", "mxb"):
            assert call(**{k: -1}) == _cabi.ERR_INVALID, (s, k)
        for k in ("n", "m"):
            assert scall(**{k: -1}) == _cabi.ERR_INVALID, (s, k)
        for ax in (-2, 3, 7):
            assert call(ax=ax) == _cabi.ERR_INVALID and call(ax=ax, nf=0) == _cabi.ERR_INVALID, (s, ax)
            assert scall(ax=ax) == _cabi.ERR_INVALID and scall(ax=ax, n=0, m=0) == _cabi.ERR_INVALID, (s, ax)
        for ax in (-1, 0, 2):   # empty problems: no work, no pointer needed
            assert call(ax=ax, nf=0) == _cabi.OK and call(ax=ax, tp=0, tb=0) == _cabi.OK, (s, ax)
            assert scall(ax=ax, n=0, m=0, p=0, b=0, pb=0, bn=0, ws=0) == _cabi.OK, (s, ax)
        assert call(nf=0, p=0, b=0, po=0, bo=0, pb=0, bn=0, ws=0) == _cabi.OK, s
        for k in ("po", "bo", "p", "b", "pb", "bn"):
            assert call(**{k: 0}) == _cabi.ERR_INVALID, (s, k)
        for k in ("p", "b", "pb", "bn"):
            assert scall(**{k: 0}) == _cabi.ERR_INVALID, (s, k)
        assert call(wsb=bw - 1) == _cabi.ERR_WORKSPACE and call(ws=0) == _cabi.ERR_WORKSPACE and call(ax=2, wsb=bw - 1) == _cabi.ERR_WORKSPACE
        assert scall(wsb=sw - 1) == _cabi.ERR_WORKSPACE and scall(ws=0) == _cabi.ERR_WORKSPACE and scall(ax=1, wsb=sw - 1) == _cabi.ERR_WORKSPACE
        assert call(nf=1 << 31) == _cabi.ERR_UNSUPPORTED, s
        assert scall(n=1 << 32) == _cabi.ERR_INVALID and scall(m=1 << 31) == _cabi.ERR_INVALID, s


def test_front_door_errors_without_gpu():
    """the exceptions of box2dr_crop / box3dp_crop and their batch forms, raised before any device work"""
    from d3d_b200.box import box2dr_crop_assign, box2dr_crop_assign_batch, box3dp_crop_assign, box3dp_crop_assign_batch
    rng = np.random.default_rng(1)
    p2, b2 = _frame(rng, 9, 4, None, np.float32)
    p3, b3 = _frame(rng, 9, 4, 2, np.float32)
    with pytest.raises(ValueError, match="Nx2"):
        box2dr_crop_assign(p3, b2)
    with pytest.raises(ValueError, match="5 fields"):
        box2dr_crop_assign(p2, b3)
    with pytest.raises(ValueError, match="Nx3"):
        box3dp_crop_assign(p2, b3)
    with pytest.raises(ValueError, match="7 fields"):
        box3dp_crop_assign(p3, b2)
    for ax in (3, -1, "z"):
        with pytest.raises(ValueError, match="projection axis"):
            box3dp_crop_assign(p3, b3, project_axis=ax)
        with pytest.raises(ValueError, match="projection axis"):
            box3dp_crop_assign_batch([p3], [b3], project_axis=ax)
    with pytest.raises(RuntimeError, match="same dtype"):
        box2dr_crop_assign(torch.from_numpy(p2), torch.from_numpy(b2.astype(np.float64)))
    with pytest.raises(RuntimeError, match="same dtype"):
        box2dr_crop_assign_batch([p2, p2], [b2, b2.astype(np.float64)])
    with pytest.raises(RuntimeError, match="float32 or float64"):
        box2dr_crop_assign(torch.from_numpy(p2).half(), torch.from_numpy(b2).half())
    with pytest.raises(ValueError, match="same number of frames"):
        box2dr_crop_assign_batch([p2, p2], [b2])
    with pytest.raises(ValueError, match="Nx2"):
        box2dr_crop_assign_batch([p2, p3], [b2, b2])
    with pytest.raises(ValueError, match="frame offsets"):
        box2dr_crop_assign_batch(p2, b2)
    with pytest.raises(ValueError, match="inconsistent"):
        box2dr_crop_assign_batch(p2, b2, np.array([0, 4, 8]), np.array([0, 2, 4]))
    with pytest.raises(ValueError, match="inconsistent"):
        box3dp_crop_assign_batch(p3, b3, np.array([0, 9]), np.array([0, 2, 4]))
    assert box2dr_crop_assign_batch([], []) == [] and box3dp_crop_assign_batch([], []) == []


# ------------------------------------------------------------------ values against the mask
@pytest.mark.gpu
@DTS
@AXES
def test_values_equal_mask_reductions(dev, dt, axis):
    """ragged frames: empty sides, 1 x 1, 15 / 16 / 17 and 4095 / 4096 / 4097 points, 15 / 16 / 17 boxes, a frame 100 km from the origin,
    a NaN point, on both back ends of the single-frame entry"""
    rng = np.random.default_rng(5)
    sizes = [(0, 5), (7, 0), (0, 0), (1, 1), (15, 7), (16, 16), (17, 15), (4095, 17), (4096, 13), (4097, 33), (300, 40)]
    frames = [_frame(rng, n, m, axis, dt) for n, m in sizes]
    frames.insert(6, _frame(rng, 500, 11, axis, dt, shift=1e5))
    p, b = _frame(rng, 40, 6, axis, dt)
    p[3] = np.nan
    p[7, -1] = np.nan
    frames.append((p, b))
    refs = _check_frames(frames, axis, dev, paths=("brute", "grid"))
    assert all(int((r[0] >= 0).sum()) > 0 for r in refs[8:12]) and int((refs[6][0] >= 0).sum()) > 0   # real hits, far from the origin too
    assert int(refs[-1][0][3]) == -1 and int(refs[-1][0][7]) == -1


@pytest.mark.gpu
@DTS
def test_golden_mask(dev, dt):
    """tests/golden/crop.npz: the outputs equal the reductions of the mask the reference's crop_2dr wrote"""
    g = golden("crop.npz")
    tag = "f32" if dt == np.float32 else "f64"
    pts, bx = g[f"{tag}.points"], g[f"{tag}.boxes"]
    exp = np.unpackbits(g[f"{tag}.mask"])[:len(bx) * len(pts)].reshape(len(bx), len(pts)).astype(bool)
    ref = _reduce(torch.from_numpy(exp))
    assert int((ref[0] >= 0).sum()) > 0 and int((ref[1] > 1).sum()) > 0
    for path in PATHS:
        try:
            _cabi.tuning_set("D3D_B200_CROP_PATH", PATHS[path])
            _eq(_assign(_t(pts, dev), _t(bx, dev), None), ref, (tag, path))
            _eq(_assign_batch([_t(pts, dev)], [_t(bx, dev)], None)[0], ref, (tag, path, "batch"))
            for axis in (0, 2):
                p3, b3 = _to3d(pts, bx, axis)
                _eq(_assign(_t(p3, dev), _t(b3, dev), axis), ref, (tag, path, axis))
        finally:
            _cabi.tuning_set("D3D_B200_CROP_PATH", None)


@pytest.mark.gpu
@DTS
@pytest.mark.parametrize("axis", [None, 1], ids=["2d", "ax1"])
def test_ties_edges_and_nan(dev, dt, axis):
    """duplicated and nested boxes (points in several boxes: the lowest index wins), points exactly on edges and vertices (open AABB,
    no negative cross product), NaN points and NaN boxes (never inside)"""
    b2 = np.array([[0, 0, 4, 4, 0], [0, 0, 2, 2, 0], [0, 0, 4, 4, 0], [0, 0, 2, 2, 0], [1, 1, 2, 2, 0], [0, 0, 2 * np.sqrt(2), 2 * np.sqrt(2), np.pi / 4],
                   [np.nan, 0, 2, 2, 0], [0, 0, np.nan, 2, 0], [0, 0, 2, 2, np.nan], [0, 0, 0, 0, 0], [0.5, 0.5, 1, 1, 0]])
    g = np.arange(-2.5, 2.51, 0.25)
    lattice = np.stack(np.meshgrid(g, g), -1).reshape(-1, 2)   # hits vertices and edges of the axis-aligned boxes exactly
    p2 = np.concatenate([lattice, [[np.nan, 0], [0, np.nan], [np.nan, np.nan], [1, 1], [1 - 1e-6, 1 - 1e-6], [2, 0], [0, 2 - 1e-6]]])
    p2, b2 = p2.astype(dt), b2.astype(dt)
    if axis is None:
        p, b = p2, b2
    else:
        p, b = _to3d(p2, b2, axis)
        p[::7, axis] = 2.5                 # exactly on the boxes' faces along the axis: outside
        b[-1, axis] = np.nan               # a box with a NaN coordinate along the axis
    refs = _check_frames([(p, b), (p[::-1].copy(), b), (p, b[::-1].copy())], axis, dev, paths=("brute", "grid"))
    pb, cnt = refs[0]
    assert int(cnt[6]) == int(cnt[7]) == int(cnt[8]) == 0 and (pb[-7:-4] == -1).all()
    assert int((pb == 1).sum()) == 0 and int((pb == 3).sum()) == 0   # every point of box 1 / 3 lies in box 0 too
    assert int(cnt[0]) == int(cnt[2]) and int(cnt[1]) == int(cnt[3]) and int(cnt[0]) > int(cnt[1]) > 0
    centre = int(np.flatnonzero((p2[:, 0] == 0) & (p2[:, 1] == 0))[0])
    assert int(pb[centre]) == 0


# ------------------------------------------------------------------ grid path
@pytest.mark.gpu
def test_grid_bench_case(dev):
    """180k lidar points x 4096 proposals (the bench crop case; boxes on the dense first metres have tens of thousands of candidates, so
    the heavy items run): brute force and grid forced, both equal to the mask's reductions"""
    from bench import lidar as bench_lidar, proposals as bench_proposals
    pts = _t(bench_lidar(300, 180_000)[:, :2].copy(), dev)
    bx = _t(bench_proposals(300, 4096, 2048)[0].astype(np.float32), dev)
    from d3d_b200.box import box2dr_crop
    ref = _reduce(box2dr_crop(pts, bx))
    assert int(ref[1].max()) > 20000 and int((ref[0] >= 0).sum()) > 1000
    for path in PATHS:
        try:
            _cabi.tuning_set("D3D_B200_CROP_PATH", PATHS[path])
            _eq(_assign(pts, bx, None), ref, path)
        finally:
            _cabi.tuning_set("D3D_B200_CROP_PATH", None)
    _eq(_assign(pts, bx, None), ref, "default")   # 737 M pairs: the grid path on its own


@pytest.mark.gpu
def test_grid_corner_cases(dev):
    """the grid path's corner cases of the mask: boxes far outside the cloud, a flat box, clustered points, a NaN point and a cloud
    without extent (both fall back to the tile kernel)"""
    rng = np.random.default_rng(17)
    pts = np.concatenate([rng.normal(0, 0.01, (5000, 2)), (rng.random((5000, 2)) - .5) * 200]).astype(np.float32)
    bx = np.array([[0, 0, 0.05, 0.05, 0.4], [1e6, 1e6, 5, 5, 0], [0, 0, 0, 3, 1], [0, 0, 400, 400, 0.1], [-90, 95, 30, 2, 2.0]], np.float32)
    nan_pts = pts.copy()
    nan_pts[17] = np.nan
    one = np.zeros((300, 2), np.float32)
    for p in (pts, nan_pts, one):
        _check_frames([(p, bx)], None, dev, paths=("grid",))
        for axis in (0, 2):
            _check_frames([_to3d(p, bx, axis)], axis, dev, paths=("grid",))


@pytest.mark.gpu
@pytest.mark.parametrize("dt,axis", [(np.float32, 2), (np.float64, 0)])
def test_grid_3d_frame(dev, dt, axis):
    """a 3-D frame above the grid threshold (16 384 points x 4 096 boxes): the plane columns are binned, the axis test runs on the
    candidates"""
    rng = np.random.default_rng(7)
    p, b = _frame(rng, 16384, 4096, axis, dt)
    assert 16384 * 4096 >= _cabi.crop_grid_min_pairs()
    refs = _check_frames([(p, b)], axis, dev)
    assert int(refs[0][1].sum()) > 1000 and int((refs[0][0] > 0).sum()) > 100


@pytest.mark.gpu
@pytest.mark.parametrize("dt,axis", [(np.float32, None), (np.float64, None), (np.float32, 2), (np.float64, 1)])
def test_mixed_batch(dev, dt, axis):
    """one call with frames on both sides of the grid threshold; the large frames' slices are written by the single-frame entry after
    the batch entry initialised every slice"""
    rng = np.random.default_rng(9)
    frames = [_frame(rng, 100, 7, axis, dt), _frame(rng, 16384, 4096, axis, dt), _frame(rng, 0, 3, axis, dt), _frame(rng, 17, 0, axis, dt),
              _frame(rng, 4097, 20, axis, dt), _frame(rng, 20000, 4000, axis, dt), _frame(rng, 5, 5, axis, dt)]
    refs = _check_frames(frames, axis, dev)
    assert int(refs[1][1].sum()) > 1000 and int(refs[5][1].sum()) > 1000
    pl, bl = [_t(p, dev) for p, _ in frames], [_t(b, dev) for _, b in frames]
    po, bo = np.cumsum([0] + [len(p) for p in pl]), np.cumsum([0] + [len(b) for b in bl])
    pb, cnt = _assign_batch(torch.cat(pl), torch.cat(bl), axis, point_offsets=po, box_offsets=bo)
    assert torch.equal(pb, torch.cat([r[0] for r in refs])) and torch.equal(cnt, torch.cat([r[1] for r in refs]))


# ------------------------------------------------------------------ scale, call forms, launches
@pytest.mark.gpu
@pytest.mark.parametrize("dt,axis", [(np.float32, None), (np.float64, 1)])
def test_over_65535_frames(dev, dt, axis):
    """70 000 frames of 1-3 points and 0-2 boxes, packed: frames on grid.x beyond 65 535"""
    rng = np.random.default_rng(11)
    nf = 70000
    ns, ms = rng.integers(1, 4, nf), rng.integers(0, 3, nf)
    A, _ = _frame(rng, int(ns.sum()), 1, axis, dt)
    _, B = _frame(rng, 1, int(ms.sum()), axis, dt)
    A[:, :2 if axis is None else 3] *= 0.3
    po, bo = np.cumsum(np.r_[0, ns]), np.cumsum(np.r_[0, ms])
    from d3d_b200.box import box2dr_crop_batch, box3dp_crop_batch
    flat, moff = (box2dr_crop_batch(_t(A, dev), _t(B, dev), po, bo) if axis is None
                  else box3dp_crop_batch(_t(A, dev), _t(B, dev), po, bo, project_axis=axis))
    pb, cnt = _assign_batch(_t(A, dev), _t(B, dev), axis, point_offsets=po, box_offsets=bo)
    pb, cnt, flat, moff = pb.cpu(), cnt.cpu(), flat.cpu(), moff.tolist()
    hits = 0
    for f in range(nf):
        r = _reduce(flat[moff[f]:moff[f + 1]].view(int(ms[f]), int(ns[f])))
        assert torch.equal(pb[po[f]:po[f + 1]], r[0]) and torch.equal(cnt[bo[f]:bo[f + 1]], r[1]), f
        hits += int(r[1].sum())
    assert hits > 20


@pytest.mark.gpu
@pytest.mark.parametrize("axis", [None, 2], ids=["2d", "ax2"])
def test_call_forms(dev, axis):
    """list vs packed (frame-local indices), numpy / host / device in and out, inputs that require grad, repeated calls identical"""
    rng = np.random.default_rng(13)
    frames = [_frame(rng, n, m, axis, np.float32) for n, m in ((300, 9), (0, 4), (50, 0), (4097, 30))]
    pn, bn = [p for p, _ in frames], [b for _, b in frames]
    po, bo = np.cumsum([0] + [len(p) for p in pn]), np.cumsum([0] + [len(b) for b in bn])
    P, B = np.concatenate(pn), np.concatenate(bn)
    ref = _assign_batch([_t(p, dev) for p in pn], [_t(b, dev) for b in bn], axis)
    assert all(x.is_cuda and y.is_cuda for x, y in ref)
    refp = (torch.cat([r[0] for r in ref]), torch.cat([r[1] for r in ref]))
    assert int(refp[0].max()) >= 9   # frame-local indices: the last frame has indices above the first frame's box count
    out = _assign_batch(pn, bn, axis)
    assert all(isinstance(x, np.ndarray) and isinstance(y, np.ndarray) for x, y in out)
    _eq((np.concatenate([o[0] for o in out]), np.concatenate([o[1] for o in out])), refp, "numpy list")
    out = _assign_batch([torch.from_numpy(p) for p in pn], [torch.from_numpy(b) for b in bn], axis)
    assert all(x.device.type == "cpu" and y.device.type == "cpu" for x, y in out)
    _eq((torch.cat([o[0] for o in out]), torch.cat([o[1] for o in out])), refp, "host list")
    out = _assign_batch(P, B, axis, point_offsets=po, box_offsets=bo)
    assert isinstance(out[0], np.ndarray)
    _eq(out, refp, "numpy packed")
    out = _assign_batch(torch.from_numpy(P), torch.from_numpy(B), axis, point_offsets=torch.from_numpy(po), box_offsets=torch.from_numpy(bo))
    assert out[0].device.type == "cpu"
    _eq(out, refp, "host packed")
    tp, tb = _t(P, dev).requires_grad_(True), _t(B, dev).requires_grad_(True)
    for _ in range(3):
        out = _assign_batch(tp, tb, axis, point_offsets=po, box_offsets=bo)
        assert not out[0].requires_grad and not out[1].requires_grad
        _eq(out, refp, "device packed, repeated")
    for f, (p, b) in enumerate(frames):
        r = (ref[f][0].cpu(), ref[f][1].cpu())
        x = _assign(p, b, axis)
        assert isinstance(x[0], np.ndarray)
        _eq(x, r, ("single numpy", f))
        x = _assign(torch.from_numpy(p), torch.from_numpy(b), axis)
        assert x[0].device.type == "cpu"
        _eq(x, r, ("single host", f))
        x = _assign(_t(p, dev).requires_grad_(True), _t(b, dev).requires_grad_(True), axis)
        assert x[0].is_cuda and not x[0].requires_grad
        _eq(x, r, ("single device", f))


@pytest.mark.gpu
@pytest.mark.parametrize("axis", [None, 0], ids=["2d", "ax0"])
def test_launch_count_independent_of_frames(dev, axis):
    """a tile-path batch costs the same launches at 2 and at 300 frames"""
    rng = np.random.default_rng(19)

    def launches(nf):
        frames = [_frame(rng, int(rng.integers(1, 2000)), int(rng.integers(1, 40)), axis, np.float32) for _ in range(nf)]
        pl, bl = [_t(p, dev) for p, _ in frames], [_t(b, dev) for _, b in frames]
        _assign_batch(pl, bl, axis)
        torch.cuda.synchronize()
        c0 = _cabi.launch_count()
        _assign_batch(pl, bl, axis)
        return _cabi.launch_count() - c0
    assert launches(2) == launches(300) == 2   # box preparation and the tile launch
