"""Frame-batched point <-> box operators (box2dr_crop_batch / box3dp_crop_batch over d3d_crop2dr_batch_*, box2dr_pdist_batch /
box3dr_pdist_batch over d3d_pdist2dr_batch_*): per frame the masks and distances equal the single-frame functions bit for bit, the
gradients agree with per-frame autograd to rounding and with the local-frame float64 references, and the call forms behave like
box3d_iou_distance_batch's."""
import ctypes as C

import numpy as np
import pytest
import torch

import pdist_cases as P
from conftest import gen_boxes, golden
from d3d_b200 import _cabi

DTS = pytest.mark.parametrize("dt", [np.float32, np.float64], ids=["f32", "f64"])
AXES = pytest.mark.parametrize("axis", [None, 0, 1, 2], ids=["2d", "ax0", "ax1", "ax2"])   # None: the 2-D functions


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda:0")


def _t(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def _bits(x):
    a = np.ascontiguousarray(x.detach().cpu().numpy() if torch.is_tensor(x) else x)
    return a.view(np.uint32 if a.dtype == np.float32 else np.uint64) if a.dtype.kind == "f" else a


def _frame(rng, n, m, axis, dt, shift=0.0):
    """n points around m boxes ([n, 2] / [m, 5], or [n, 3] / [m, 7] for a projection axis), moved by `shift` metres"""
    b2 = gen_boxes(rng, m) + [0, 0, .2, .2, 0]
    p2 = (rng.random((n, 2)) - .5) * 12
    if axis is None:
        b, p = b2, p2
    else:   # x, y, z, lx, ly, lz, r with the BEV box in the two columns other than the axis
        b = np.zeros((m, 7))
        pc, bc = {0: ([1, 2], [1, 2, 4, 5, 6]), 1: ([0, 2], [0, 2, 3, 5, 6]), 2: ([0, 1], [0, 1, 3, 4, 6])}[axis]
        b[:, bc] = b2
        b[:, axis], b[:, 3 + axis] = rng.normal(0, 1, m), 0.5 + rng.random(m) * 3
        p = np.zeros((n, 3))
        p[:, pc] = p2
        p[:, axis] = (rng.random(n) - .5) * 5
    p, b = p + shift, b.copy()
    b[:, :2 if axis is None else 3] += shift
    return p.astype(dt), b.astype(dt)


# ------------------------------------------------------------------ C ABI, no GPU needed
def test_cabi_argument_errors_without_gpu():
    """argument errors return codes before any CUDA call; empty batches are a no-op"""
    lib = C.CDLL(_cabi.LIB_PATH)
    i64, vp, sz = C.c_int64, C.c_void_p, C.c_size_t
    gmp = lib.d3d_crop2dr_grid_min_pairs
    gmp.restype = i64
    assert gmp() == 64 << 20
    wsb = lib.d3d_crop2dr_batch_workspace_bytes
    wsb.restype, wsb.argtypes = sz, [i64, C.c_int]
    need = wsb(20, 0)
    assert need >= 20 * 48 and wsb(20, 1) >= 20 * 96 and wsb(-1, 0) == 0
    names = ["p", "tp", "po", "b", "tb", "bo", "nf", "mxp", "mxb", "ax", "oo", "out"]
    crop = lib.d3d_crop2dr_batch_f32
    crop.argtypes = [vp, i64, vp, vp, i64, vp, i64, i64, i64, C.c_int, vp, vp, vp, sz, vp]
    pd = lib.d3d_pdist2dr_batch_f64
    pd.argtypes = [vp, i64, vp, vp, i64, vp, i64, i64, i64, C.c_int, vp, vp, vp]
    bw = lib.d3d_pdist2dr_batch_backward_f32
    bw.argtypes = [vp, i64, vp, vp, i64, vp, i64, i64, i64, C.c_int, vp, vp, vp, vp, vp]
    ok = [8, 30, 8, 8, 20, 8, 3, 16, 9, -1, 8, 8]
    calls = {"crop": (crop, names + ["ws", "wsb", "st"], ok + [8, need, 0]), "pdist": (pd, names + ["st"], ok + [0]),
             "backward": (bw, names + ["gb", "gp", "st"], ok + [8, 8, 0])}
    for what, (fn, keys, base) in calls.items():
        def call(**kw):
            a = list(base)
            for k, v in kw.items():
                a[keys.index(k)] = v
            return fn(*a)
        for k in ("tp", "tb", "nf", "mxp", "mxb"):
            assert call(**{k: -1}) == _cabi.ERR_INVALID, (what, k)
        for ax in (-2, 3, 7):
            assert call(ax=ax) == _cabi.ERR_INVALID and call(ax=ax, nf=0) == _cabi.ERR_INVALID, (what, ax)
        for ax in (-1, 0, 2):
            assert call(ax=ax, nf=0) == _cabi.OK and call(ax=ax, tp=0) == _cabi.OK and call(ax=ax, tb=0) == _cabi.OK, (what, ax)
        assert call(nf=0, p=0, b=0, po=0, bo=0, oo=0, out=0) == _cabi.OK, what
        for k in ("po", "bo", "oo", "p", "b", "out"):
            assert call(**{k: 0}) == _cabi.ERR_INVALID, (what, k)
    call = lambda **kw: crop(*[kw.get(k, v) for k, v in zip(names + ["ws", "wsb", "st"], ok + [8, need, 0])])  # noqa: E731
    assert call(wsb=need - 1) == _cabi.ERR_WORKSPACE and call(ws=0) == _cabi.ERR_WORKSPACE
    assert call(ax=2, wsb=need - 1) == _cabi.ERR_WORKSPACE
    bcall = lambda **kw: bw(*[kw.get(k, v) for k, v in zip(names + ["gb", "gp", "st"], ok + [8, 8, 0])])  # noqa: E731
    assert bcall(gb=0) == _cabi.ERR_INVALID and bcall(gp=0) == _cabi.ERR_INVALID


# ------------------------------------------------------------------ masks
def _single_crop(p, b, axis):
    from d3d_b200.box import box2dr_crop, box3dp_crop
    return box2dr_crop(p, b) if axis is None else box3dp_crop(p, b, project_axis=axis)


def _batch_crop(pl, bl, axis, **kw):
    from d3d_b200.box import box2dr_crop_batch, box3dp_crop_batch
    return box2dr_crop_batch(pl, bl, **kw) if axis is None else box3dp_crop_batch(pl, bl, project_axis=axis, **kw)


def _check_crop_frames(frames, axis, dev, sample=None):
    blocks = _batch_crop([_t(p, dev) for p, _ in frames], [_t(b, dev) for _, b in frames], axis)
    assert len(blocks) == len(frames)
    for f in (range(len(frames)) if sample is None else sample):
        p, b = frames[f]
        blk = blocks[f]
        assert blk.is_cuda and blk.dtype == torch.bool and tuple(blk.shape) == (len(b), len(p)), f
        assert torch.equal(blk, _single_crop(_t(p, dev), _t(b, dev), axis)), (axis, f, len(p), len(b))
    return blocks


def _golden_frame(dt, axis):
    """the golden crop.npz frame; 3-D: the same BEV boxes with every point inside the boxes' extent along the axis"""
    g = golden("crop.npz")
    tag = "f32" if dt == np.float32 else "f64"
    pts, bx = g[f"{tag}.points"], g[f"{tag}.boxes"]
    exp = np.unpackbits(g[f"{tag}.mask"])[:len(bx) * len(pts)].reshape(len(bx), len(pts)).astype(bool)
    if axis is None:
        return pts, bx, exp
    pc, bc = {0: ([1, 2], [1, 2, 4, 5, 6]), 1: ([0, 2], [0, 2, 3, 5, 6]), 2: ([0, 1], [0, 1, 3, 4, 6])}[axis]
    p, b = np.zeros((len(pts), 3), dt), np.zeros((len(bx), 7), dt)
    p[:, pc], b[:, bc] = pts, bx
    p[:, axis], b[:, axis], b[:, 3 + axis] = 0.25, 0.5, 4
    return p, b, exp


@pytest.mark.gpu
@DTS
@AXES
def test_crop_batch_bit_equal_per_frame(dev, dt, axis):
    """empty sides, 1 x 1, N_f of 1, 15, 16, 17 and 4097 with odd block offsets, a frame 100 km from the origin, a NaN point, and the
    golden crop frame packed between two others"""
    rng = np.random.default_rng(5)
    sizes = [(0, 5), (7, 0), (0, 0), (1, 1), (1, 3), (15, 7), (16, 5), (17, 9), (4097, 13), (33, 16), (300, 17)]
    frames = [_frame(rng, n, m, axis, dt) for n, m in sizes]
    frames.insert(6, _frame(rng, 500, 11, axis, dt, shift=1e5))
    p, b = _frame(rng, 40, 6, axis, dt)
    p[3] = np.nan
    p[7, -1] = np.nan
    frames.append((p, b))
    gp, gb, exp = _golden_frame(dt, axis)
    frames += [_frame(rng, 70, 5, axis, dt), (gp, gb), _frame(rng, 9, 31, axis, dt)]
    blocks = _check_crop_frames(frames, axis, dev)
    assert np.array_equal(blocks[-2].cpu().numpy(), exp)
    assert blocks[-2].any() and blocks[6].any() and blocks[9].any()   # real hits, far from the origin too
    assert not blocks[-4][:, 3].any() and not blocks[-4][:, 7].any()  # NaN points are outside every box


@pytest.mark.gpu
@pytest.mark.parametrize("dt,axis", [(np.float32, None), (np.float64, None), (np.float32, 2), (np.float64, 0)])
def test_crop_batch_frame_above_grid_threshold(dev, dt, axis):
    """a frame of 16 384 points x 4 096 boxes (64 M pairs, the single-frame grid path) between small frames"""
    from d3d_b200 import _cabi as _c
    rng = np.random.default_rng(7)
    assert 16384 * 4096 >= _c.crop_grid_min_pairs()
    big = _frame(rng, 16384, 4096, axis, dt)
    frames = [_frame(rng, 100, 7, axis, dt), big, _frame(rng, 17, 3, axis, dt), _frame(rng, 4097, 20, axis, dt)]
    blocks = _check_crop_frames(frames, axis, dev)
    assert int(blocks[1].sum()) > 1000


@pytest.mark.gpu
@pytest.mark.parametrize("dt,axis", [(np.float32, None), (np.float64, 1)])
def test_crop_batch_over_65535_frames(dev, dt, axis):
    """70 000 frames of 1-3 points and 0-2 boxes, packed: frames on grid.x beyond 65 535"""
    rng = np.random.default_rng(11)
    nf = 70000
    ns, ms = rng.integers(1, 4, nf), rng.integers(0, 3, nf)
    A, _ = _frame(rng, int(ns.sum()), 1, axis, dt)
    _, B = _frame(rng, 1, int(ms.sum()), axis, dt)
    A[:, :2 if axis is None else 3] *= 0.3
    po, bo = np.cumsum(np.r_[0, ns]), np.cumsum(np.r_[0, ms])
    flat, moff = _batch_crop(_t(A, dev), _t(B, dev), axis, point_offsets=po, box_offsets=bo)
    assert moff.tolist() == np.cumsum(np.r_[0, ns * ms]).tolist()
    sample = list(range(0, nf, 251)) + list(range(65530, 65541)) + list(range(nf - 100, nf))
    hits = 0
    for f in sample:
        blk = flat[int(moff[f]):int(moff[f + 1])].view(int(ms[f]), int(ns[f]))
        assert torch.equal(blk, _single_crop(_t(A[po[f]:po[f + 1]], dev), _t(B[bo[f]:bo[f + 1]], dev), axis)), f
        hits += int(blk.sum())
    assert hits > 20


# ------------------------------------------------------------------ distances
def _single_pdist(p, b, axis):
    from d3d_b200.box import box2dr_pdist, box3dr_pdist
    return box2dr_pdist(p, b) if axis is None else box3dr_pdist(p, b, project_axis=axis)


def _batch_pdist(pl, bl, axis, **kw):
    from d3d_b200.box import box2dr_pdist_batch, box3dr_pdist_batch
    return box2dr_pdist_batch(pl, bl, **kw) if axis is None else box3dr_pdist_batch(pl, bl, project_axis=axis, **kw)


def _leaf(a, dev):
    return _t(a, dev).requires_grad_(True)


def _check_pdist_frames(frames, axis, dev, dt):
    """values bit for bit and both gradients to rounding against per-frame autograd; returns the batch's (values, point grads, box grads)"""
    tol = 1e-4 if dt == np.float32 else 1e-12
    rng = np.random.default_rng(99)
    ups = [rng.normal(size=(len(b), len(p))).astype(dt) for p, b in frames]
    pl, bl = [_leaf(p, dev) for p, _ in frames], [_leaf(b, dev) for _, b in frames]
    blocks = _batch_pdist(pl, bl, axis)
    sum((blk * _t(u, dev)).sum() for blk, u in zip(blocks, ups)).backward()
    for f, ((p, b), u) in enumerate(zip(frames, ups)):
        sp, sb = _leaf(p, dev), _leaf(b, dev)
        v = _single_pdist(sp, sb, axis)
        assert blocks[f].dtype == v.dtype and blocks[f].shape == v.shape, f
        assert np.array_equal(_bits(blocks[f]), _bits(v)), (axis, f, len(p), len(b))
        if v.numel():
            (v * _t(u, dev)).sum().backward()
            assert P.rel_err(pl[f].grad.cpu().numpy(), sp.grad.cpu().numpy().astype(np.float64)) <= tol, (axis, f)
            assert P.rel_err(bl[f].grad.cpu().numpy(), sb.grad.cpu().numpy().astype(np.float64)) <= tol, (axis, f)
    return blocks, [x.grad for x in pl], [x.grad for x in bl]


@pytest.mark.gpu
@DTS
@AXES
def test_pdist_batch_equal_per_frame(dev, dt, axis):
    """values bit for bit, gradients to rounding: empty sides, 1 x 1, tile edges (255 / 256 / 257 points, 7 / 8 / 9 boxes), a frame moved
    1 km (fp32) or 100 km (fp64) from the origin"""
    rng = np.random.default_rng(13)
    sizes = [(0, 4), (6, 0), (1, 1), (255, 7), (256, 8), (257, 9), (40, 12), (600, 30)]
    frames = [_frame(rng, n, m, axis, dt) for n, m in sizes]
    frames.insert(3, _frame(rng, 120, 10, axis, dt, shift=1e3 if dt == np.float32 else 1e5))
    blocks, _, _ = _check_pdist_frames(frames, axis, dev, dt)
    assert (blocks[-1] > 0).any() and (blocks[-1] < 0).any()


def _grad5(fn, x, cols, h):
    """five-point derivative of fn (values [M, N]) in every column of `cols` of x, all rows moved at once: [len(cols), M, N]"""
    out = []
    for c in cols:
        def at(s):
            y = x.copy()
            y[:, c] += s
            return fn(y)
        out.append((8 * (at(h) - at(-h)) - (at(2 * h) - at(-2 * h))) / (12 * h))
    return np.stack(out)


def _oracle_grads(oracle, p, b, axis, up, h=1e-4):
    """(value, grad points, grad boxes, upstream with the non-smooth pairs zeroed) of oracle.pdist2dr_local / box3dr_pdist_local: a pair
    is smooth when the stencils at h and h / 2 agree to 1e-9"""
    f = (lambda pp, bb: oracle.pdist2dr_local(pp, bb)) if axis is None else (lambda pp, bb: oracle.box3dr_pdist_local(pp, bb, axis))
    pc, bc = range(p.shape[1]), range(b.shape[1])
    dp, db = _grad5(lambda y: f(y, b), p, pc, h), _grad5(lambda y: f(p, y), b, bc, h)
    dp2, db2 = _grad5(lambda y: f(y, b), p, pc, h / 2), _grad5(lambda y: f(p, y), b, bc, h / 2)
    smooth = (np.abs(dp - dp2).max(0) < 1e-9) & (np.abs(db - db2).max(0) < 1e-9)
    u = np.where(smooth, up, 0)
    return f(p, b), np.einsum("ij,cij->jc", u, dp), np.einsum("ij,cij->ic", u, db), u, smooth


@pytest.mark.gpu
@AXES
def test_pdist_batch_vs_local_reference(dev, oracle, axis):
    """fp64 values and gradients against the local-frame float64 references and their five-point differences, the case frame packed
    between two others; the 2-D shared cases of pdist_cases (headings, zero-size boxes, translation) run through the batch"""
    rng = np.random.default_rng(17)
    p, b = _frame(rng, 80, 9, axis, np.float64)
    up = rng.normal(size=(9, 80))
    v, gp, gb, u, smooth = _oracle_grads(oracle, p, b, axis, up)
    assert smooth.mean() > 0.8
    frames = [_frame(rng, 30, 4, axis, np.float64), (p, b), _frame(rng, 5, 3, axis, np.float64)]
    pl, bl = [_leaf(x, dev) for x, _ in frames], [_leaf(x, dev) for _, x in frames]
    blocks = _batch_pdist(pl, bl, axis)
    (blocks[1] * _t(u, dev)).sum().backward()
    assert P.val_err(blocks[1].detach().cpu().numpy(), v) <= 1e-10
    assert P.rel_err(pl[1].grad.cpu().numpy(), gp) <= 1e-8 and P.rel_err(bl[1].grad.cpu().numpy(), gb) <= 1e-8
    assert not pl[0].grad.any() and not bl[2].grad.any()   # the other frames got no gradient from this one
    if axis is not None:
        return

    def run(points, boxes, upm):
        other = _frame(np.random.default_rng(1), 7, 2, None, points.dtype)
        tp, tb = [_leaf(other[0], dev), _leaf(points, dev)], [_leaf(other[1], dev), _leaf(boxes, dev)]
        out = _batch_pdist(tp, tb, None)
        (out[1] * _t(upm, dev)).sum().backward()
        return out[1].detach().cpu().numpy(), None, tp[1].grad.cpu().numpy(), tb[1].grad.cpu().numpy()
    for dt in (np.float32, np.float64):
        P.check_headings(run, oracle, dt)
        P.check_zero_size(run, oracle, dt)
        P.check_edge_lines(run, oracle, dt)
        vt, gt = P.TOL[dt]
        for off in P.OFFSETS[dt]:
            tp_, tb_, up_ = P.translation_case(off, dt)
            rv, rgp, rgb, upm, _ = P.reference(oracle, tp_, tb_, up_)
            kv, _, kp, kb = run(tp_, tb_, upm)
            assert P.val_err(kv, rv) <= vt and P.rel_err(kp, rgp) <= gt and P.rel_err(kb, rgb) <= gt, (dt, off)


@pytest.mark.gpu
@DTS
def test_pdist3d_tie_and_prism_edges(dev, dt):
    """dyadic inputs: d2 == dp > 0 gives each term half of the gradient (torch.minimum's rule), exactly; points on the edges of the prism
    (d2 = dp = 0) get finite gradients, as in box3dr_pdist"""
    box = np.array([[0.5, -0.25, 0.0, 4, 2, 2, 0]], dt)
    tie = np.array([[0.5, -0.25, 0.0], [1.0, -0.25, 0.25]], dt)   # d2 = dp = 1 (a tie); d2 = 1 > dp = 0.75
    pl, bl = [_leaf(tie, dev)], [_leaf(box, dev)]
    d = _batch_pdist(pl, bl, 2)[0]
    assert d.detach().cpu().numpy().tolist() == [[1.0, 0.75]]
    d.sum().backward()
    gp, gb = pl[0].grad.cpu().numpy(), bl[0].grad.cpu().numpy()
    # point 0 (the centre): d2 = h/2 + qy (edge 0 is the first of the two as near) and dp = p - (c - d/2), half each; point 1: dp = c + d/2 - p
    assert gp.tolist() == [[0, 0.5, 0.5], [0, 0, -1]]
    assert gb.tolist() == [[0, -0.5, -0.5 + 1, 0, 0.5 * 0.5, 0.5 * 0.5 + 0.5, 0]]
    sp, sb = _leaf(tie, dev), _leaf(box, dev)
    _single_pdist(sp, sb, 2).sum().backward()
    assert np.array_equal(gp, sp.grad.cpu().numpy()) and np.array_equal(gb, sb.grad.cpu().numpy())
    # prism edges and corners: on the BEV boundary at z = c +- d/2, and BEV corners
    b = np.array([[0, 0, 0, 4, 2, 2, 0.3], [1, 1, 1, 2, 2, 2, 0]], dt)
    c, s = np.cos(0.3), np.sin(0.3)
    local = np.array([[2, 0], [0, 1], [-2, 0.5], [2, 1], [-1, -1]])
    xy = np.stack([c * local[:, 0] - s * local[:, 1], s * local[:, 0] + c * local[:, 1]], 1)
    pts = np.concatenate([np.c_[xy, np.full(5, 1.0)], np.c_[xy, np.full(5, -1.0)], [[2, 2, 2], [0, 1, 0], [2, 1, 1.5]]]).astype(dt)
    pl, bl = [_leaf(pts, dev)], [_leaf(b, dev)]
    d = _batch_pdist(pl, bl, 2)[0]
    (d * torch.ones_like(d)).sum().backward()
    assert torch.isfinite(pl[0].grad).all() and torch.isfinite(bl[0].grad).all()
    assert np.array_equal(_bits(d), _bits(_single_pdist(_t(pts, dev), _t(b, dev), 2)))


@pytest.mark.gpu
def test_pdist3d_rejects_non_positive_extent(dev):
    from d3d_b200.box import box3dr_pdist_batch
    rng = np.random.default_rng(19)
    for axis in (0, 1, 2):
        frames = [_frame(rng, 10, 3, axis, np.float64) for _ in range(3)]
        frames[1][1][2, 3 + axis] = 0.0
        with pytest.raises(AssertionError):
            box3dr_pdist_batch([_t(p, dev) for p, _ in frames], [_t(b, dev) for _, b in frames], project_axis=axis)
        frames[1][1][2, 3 + axis] = -1.0
        with pytest.raises(AssertionError):
            box3dr_pdist_batch([p for p, _ in frames], [b for _, b in frames], project_axis=axis)


# ------------------------------------------------------------------ call forms
@pytest.mark.gpu
@pytest.mark.parametrize("op", ["crop2d", "crop3d", "pdist2d", "pdist3d"])
def test_call_forms(dev, op):
    """list and packed forms agree; numpy in -> numpy out; host tensors in -> host tensors out; non-contiguous inputs; the argument
    errors of the single-frame functions"""
    from d3d_b200 import box as B
    axis = None if op.endswith("2d") else 1
    fn = {"crop2d": B.box2dr_crop_batch, "crop3d": B.box3dp_crop_batch, "pdist2d": B.box2dr_pdist_batch, "pdist3d": B.box3dr_pdist_batch}[op]
    kw = {} if axis is None else dict(project_axis=axis)
    rng = np.random.default_rng(23)
    sizes = [(40, 7), (0, 3), (17, 9), (5, 0), (300, 11)]
    fr = [_frame(rng, n, m, axis, np.float64) for n, m in sizes]
    po, bo = np.cumsum([0] + [n for n, _ in sizes]), np.cumsum([0] + [m for _, m in sizes])
    A, Bx = np.concatenate([p for p, _ in fr]), np.concatenate([b for _, b in fr])

    lst = fn([_t(p, dev) for p, _ in fr], [_t(b, dev) for _, b in fr], **kw)
    flat, off = fn(_t(A, dev), _t(Bx, dev), torch.from_numpy(po), torch.from_numpy(bo), **kw)
    assert flat.is_cuda and off.device.type == "cpu" and off.tolist() == np.cumsum([0] + [n * m for n, m in sizes]).tolist()
    assert np.array_equal(_bits(flat), _bits(torch.cat([x.reshape(-1) for x in lst])))
    assert all(x.untyped_storage().data_ptr() == lst[0].untyped_storage().data_ptr() for x in lst)   # views into one buffer
    assert all(tuple(x.shape) == (m, n) for x, (n, m) in zip(lst, sizes))
    flat_np, off_np = fn(A, Bx, po, bo, **kw)
    assert isinstance(flat_np, np.ndarray) and isinstance(off_np, np.ndarray) and np.array_equal(_bits(flat_np), _bits(flat))
    lst_np = fn([p for p, _ in fr], [b for _, b in fr], **kw)
    assert all(isinstance(x, np.ndarray) and x.shape == (m, n) for x, (n, m) in zip(lst_np, sizes))
    flat_cpu, _ = fn(torch.from_numpy(A), torch.from_numpy(Bx), po, bo, **kw)
    assert flat_cpu.device.type == "cpu" and np.array_equal(_bits(flat_cpu), _bits(flat))
    # non-contiguous: every other row of a doubled array, and a transposed copy
    A2, B2 = _t(np.repeat(A, 2, 0), dev)[::2], _t(np.ascontiguousarray(Bx.T), dev).t()
    assert not A2.is_contiguous() and not B2.is_contiguous()
    flat_nc, _ = fn(A2, B2, po, bo, **kw)
    assert np.array_equal(_bits(flat_nc), _bits(flat))
    assert fn([], [], **kw) == []
    f0, o0 = fn(torch.zeros((0, A.shape[1]), dtype=torch.float64), torch.zeros((0, Bx.shape[1]), dtype=torch.float64), [0], [0], **kw)
    assert f0.numel() == 0 and o0.tolist() == [0]
    bad_p, bad_b = np.zeros((4, A.shape[1] + 1)), np.zeros((2, Bx.shape[1]))
    with pytest.raises(ValueError, match="Input points should be"):
        fn([bad_p], [bad_b], **kw)
    with pytest.raises(ValueError, match="fields"):
        fn([np.zeros((4, A.shape[1]))], [np.zeros((2, Bx.shape[1] - 1))], **kw)
    with pytest.raises(ValueError):
        fn(A, Bx, po[:-1], bo[:-1], **kw)
    with pytest.raises(ValueError):
        fn(A, Bx, **kw)
    with pytest.raises(RuntimeError):
        fn([_t(A, dev).float()], [_t(Bx, dev)], **kw)
    if axis is not None:
        with pytest.raises(ValueError, match="projection axis"):
            fn(A, Bx, po, bo, project_axis=3)
    if op.startswith("pdist"):   # list-form autograd reaches every per-frame input
        pl, bl = [_leaf(p, dev) for p, _ in fr], [_leaf(b, dev) for _, b in fr]
        sum(x.sum() for x in fn(pl, bl, **kw)).backward()
        for (p, b), gp, gb in zip(fr, pl, bl):
            assert gp.grad is not None and gb.grad is not None and gp.grad.shape == gp.shape and gb.grad.shape == gb.shape
            sp, sb = _leaf(p, dev), _leaf(b, dev)
            v = _single_pdist(sp, sb, axis)
            if v.numel():
                v.sum().backward()
                assert P.rel_err(gp.grad.cpu().numpy(), sp.grad.cpu().numpy()) <= 1e-12 and P.rel_err(gb.grad.cpu().numpy(), sb.grad.cpu().numpy()) <= 1e-12
    torch.cuda.synchronize()
