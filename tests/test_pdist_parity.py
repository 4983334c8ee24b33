"""The signed point-to-box distance (box2dr_pdist / box3dr_pdist, dist.cu) against the local-frame float64 reference
(oracle.pdist2dr_local / pdist2dr_grad_local / box3dr_pdist_local): values, edge indices and both gradients in fp64 and fp32 -- the
checks of test_pdist_twin.py on the kernels -- and the shapes of the backward, box counts past one grid row of tiles, the 3-D wrapper
and empty, host-tensor and non-contiguous calls.  Needs a B200: run with `pytest -m gpu`."""
import numpy as np
import pytest
import torch

import pdist_cases as P
from conftest import gen_boxes

pytestmark = pytest.mark.gpu
DTS = pytest.mark.parametrize("dt", [np.float32, np.float64], ids=["f32", "f64"])


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda:0")


def _t(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def edges(tp, tb):
    """(value, edge index) [M, N] of the C ABI's forward with an edge buffer"""
    from d3d_b200 import _cabi as _c
    n, m = tp.shape[0], tb.shape[0]
    d = torch.empty((m, n), dtype=tp.dtype, device=tp.device)
    e = torch.full((m, n), 255, dtype=torch.uint8, device=tp.device)
    st = _c.pdist2dr[_c.dtype_code(tp.dtype)](_c.ptr(tp), n, _c.ptr(tb), m, _c.ptr(d), _c.ptr(e), _c.stream_ptr())
    assert st == _c.OK, _c.error_string(st)
    return d, e


@pytest.fixture(scope="module")
def run(dev):
    from d3d_b200.box import box2dr_pdist

    def f(points, boxes, up):
        tp, tb = _t(points, dev).requires_grad_(True), _t(boxes, dev).requires_grad_(True)
        v = box2dr_pdist(tp, tb)
        (v * _t(up, dev)).sum().backward()
        d, e = edges(tp.detach(), tb.detach())
        assert torch.equal(d, v.detach())
        return v.detach().cpu().numpy(), e.cpu().numpy(), tp.grad.cpu().numpy(), tb.grad.cpu().numpy()
    return f


@DTS
def test_translation(run, oracle, dt):
    print(dt.__name__, P.check_translation(run, oracle, dt))


@DTS
def test_edge_lines(run, oracle, dt):
    P.check_edge_lines(run, oracle, dt)


def test_ties(run, oracle):
    P.check_ties(run, oracle)


@DTS
def test_headings(run, oracle, dt):
    P.check_headings(run, oracle, dt)


def test_equivalent_boxes(run):
    P.check_equivalent_boxes(run)


@DTS
def test_zero_size(run, oracle, dt):
    P.check_zero_size(run, oracle, dt)


def test_lidar_scene(run, oracle):
    P.check_lidar_scene(run, oracle)


@DTS
def test_backward_shapes(run, oracle, dt):
    """n points over 1, 31, 32, 33, 255, 256, 257 (256 per CTA, partial warps) x m boxes over 1, 7, 8, 9, 17 (8 per CTA): against the
    reference, and against the sums of the same backward over point chunks (box gradients) and box chunks (point gradients)"""
    vt, gt = P.TOL[dt]
    rng = np.random.default_rng(51)
    for n in (1, 31, 32, 33, 255, 256, 257):
        for m in (1, 7, 8, 9, 17):
            b = (gen_boxes(rng, m) + [0, 0, .2, .2, 0]).astype(dt)
            p = P.near_points(rng, b.astype(np.float64), n).astype(dt)
            up = rng.normal(size=(m, n)).astype(dt)
            v, gp, gb, upm, _ = P.reference(oracle, p, b, up)
            kv, _, kp, kb = run(p, b, upm)
            e = (P.val_err(kv, v), P.rel_err(kp, gp), P.rel_err(kb, gb))
            assert e[0] <= vt and e[1] <= gt and e[2] <= gt, (n, m, e)
            sp = sum(run(p, b[c:c + 3], upm[c:c + 3])[2].astype(np.float64) for c in range(0, m, 3))
            sb = sum(run(p[c:c + 40], b, upm[:, c:c + 40])[3].astype(np.float64) for c in range(0, n, 40))
            ct = 1e-4 if dt == np.float32 else 1e-12   # the atomics add in another order
            assert P.rel_err(kp, sp) <= ct and P.rel_err(kb, sb) <= ct, (n, m)


def test_large_calls(run, oracle, dev):
    """524 281 boxes (65 536 tiles of 8, past one grid row of 65 535) x 3 points, and 2^20 + 3 points x 9 boxes: values on every pair,
    gradients on the first and last rows / points against the reference and the box gradients against sums over point chunks"""
    from d3d_b200.box import box2dr_pdist
    rng = np.random.default_rng(53)
    b = gen_boxes(rng, 524281, spread=40.0) + [0, 0, .2, .2, 0]
    p = (rng.random((3, 2)) - .5) * 40
    up = rng.normal(size=(len(b), 3))
    kv, _, kp, kb = run(p, b, up)
    assert P.val_err(kv, oracle.pdist2dr_local(p, b)) <= 1e-10
    rows = np.r_[0:9, 524272:524281]
    _, _, gb, upm, smooth = P.reference(oracle, p, b[rows], up[rows])
    ok = smooth.all(1)
    assert ok.mean() > 0.5 and P.rel_err(kb[rows][ok], gb[ok]) <= 1e-8
    b = gen_boxes(rng, 9) + [0, 0, .2, .2, 0]
    p = P.near_points(rng, b, (1 << 20) + 3)
    up = rng.normal(size=(9, len(p)))
    kv, _, kp, kb = run(p, b, up)
    assert P.val_err(kv, oracle.pdist2dr_local(p, b)) <= 1e-10
    cols = np.r_[0:300, len(p) - 300:len(p)]
    _, gp, _, upm, smooth = P.reference(oracle, p[cols], b, up[:, cols])
    assert P.rel_err(kp[cols][smooth.all(0)], gp[smooth.all(0)]) <= 1e-8
    tb = _t(b, dev)
    sb = torch.zeros_like(tb)
    for c in range(0, len(p), 1 << 18):
        tbc = tb.clone().requires_grad_(True)
        (box2dr_pdist(_t(p[c:c + (1 << 18)], dev), tbc) * _t(up[:, c:c + (1 << 18)], dev)).sum().backward()
        sb += tbc.grad
    assert P.rel_err(kb, sb.cpu().numpy()) <= 1e-10


def _grad3d_local(oracle, p, b, ax, h=1e-4, tol=1e-9):
    """(d value / d points [M, N, 3], d value / d boxes [M, N, 7], smooth [M, N]) of oracle.box3dr_pdist_local by five-point differences"""
    out, smooth = [], np.ones((len(b), len(p)), bool)
    for side, k in [(0, k) for k in range(3)] + [(1, k) for k in range(7)]:
        est = []
        for hh in (h, h / 2):
            f = []
            for s in (-2, -1, 1, 2):
                p_, b_ = p.copy(), b.copy()
                (b_ if side else p_)[:, k] += s * hh
                f.append(oracle.box3dr_pdist_local(p_, b_, ax))
            est.append((f[0] - 8 * f[1] + 8 * f[2] - f[3]) / (12 * hh))
        out.append(est[0])
        smooth &= np.abs(est[0] - est[1]) <= tol
    d = np.stack(out, -1)
    return d[..., :3], d[..., 3:], smooth


def test_box3dr_pdist(dev, oracle):
    """values and autograd gradients of the 3-D wrapper on all three projection axes against the local reference, and finite
    gradients for points on the edges of a box, where both the 2-D and the 1-D distance are 0"""
    from d3d_b200.box import box3dr_pdist
    rng = np.random.default_rng(55)
    b3 = np.concatenate([gen_boxes(rng, 12)[:, :2], rng.random((12, 1)), rng.random((12, 3)) * 4 + .2, rng.random((12, 1)) * 6], 1)
    p3 = b3[rng.integers(0, 12, 300), :3] + (rng.random((300, 3)) - .5) * 6
    up = rng.normal(size=(12, 300))
    for ax in (0, 1, 2):
        dp, db, smooth = _grad3d_local(oracle, p3, b3, ax)
        upm = up * smooth
        tp, tb = _t(p3, dev).requires_grad_(True), _t(b3, dev).requires_grad_(True)
        v = box3dr_pdist(tp, tb, ax)
        (v * _t(upm, dev)).sum().backward()
        assert smooth.mean() > 0.95, ax
        assert P.val_err(v.detach().cpu().numpy(), oracle.box3dr_pdist_local(p3, b3, ax)) <= 1e-10, ax
        assert P.rel_err(tp.grad.cpu().numpy(), np.einsum("ij,ijk->jk", upm, dp)) <= 1e-8, ax
        assert P.rel_err(tb.grad.cpu().numpy(), np.einsum("ij,ijk->ik", upm, db)) <= 1e-8, ax
    box = np.array([[0.5, -1, 0.25, 4, 2, 2, 0]])   # heading 0 and dyadic coordinates: both distances are exactly 0 on the edges
    p = box[:, :3] + np.array([[2, 0.25, 1], [-2, -1, -1], [0.75, 1, 1], [2, 1, 0.25], [2, 1, 1], [-1.5, -1, 1]])
    tp, tb = _t(p, dev).requires_grad_(True), _t(box, dev).requires_grad_(True)
    v = box3dr_pdist(tp, tb, 2)
    v.sum().backward()
    assert np.abs(v.detach().cpu().numpy()).max() < 1e-12
    assert bool(torch.isfinite(tp.grad).all()) and bool(torch.isfinite(tb.grad).all())


def test_calls(dev, oracle):
    """an empty side (zero gradients), host tensors in and out, non-contiguous points and a transposed upstream gradient"""
    from d3d_b200.box import box2dr_pdist
    rng = np.random.default_rng(57)
    b = gen_boxes(rng, 6)
    p = P.near_points(rng, b, 50)
    for x, y in ((p, np.zeros((0, 5))), (np.zeros((0, 2)), b)):
        tx, ty = _t(x, dev).requires_grad_(True), _t(y, dev).requires_grad_(True)
        v = box2dr_pdist(tx, ty)
        assert v.shape == (len(y), len(x))
        v.sum().backward()
        assert torch.equal(tx.grad, torch.zeros_like(tx)) and torch.equal(ty.grad, torch.zeros_like(ty))
    hv = box2dr_pdist(torch.from_numpy(p.astype(np.float32)), torch.from_numpy(b.astype(np.float32)))
    assert hv.device.type == "cpu" and P.val_err(hv.numpy(), oracle.pdist2dr_local(p.astype(np.float32), b.astype(np.float32))) <= 1e-5
    up = rng.normal(size=(6, 50))
    v, gp, gb, upm, _ = P.reference(oracle, p, b, up)
    wide = _t(np.concatenate([p[:, :1], rng.random((50, 3)), p[:, 1:]], 1), dev)
    tp = wide[:, [0, 4]].detach().requires_grad_(True)
    pv = wide[:, ::4]                                              # a strided view of the same points
    assert not pv.is_contiguous()
    tb = _t(b, dev).requires_grad_(True)
    assert torch.equal(box2dr_pdist(pv, tb).detach(), box2dr_pdist(tp, tb).detach())
    (box2dr_pdist(tp, tb).t() * _t(upm.T, dev)).sum().backward()   # the upstream gradient reaches the backward as a transposed view
    assert P.rel_err(tp.grad.cpu().numpy(), gp) <= 1e-8 and P.rel_err(tb.grad.cpu().numpy(), gb) <= 1e-8
