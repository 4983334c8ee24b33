"""The differentiable IoU family (box2d_iou "box" / "rbox" / "grbox" / "drbox", iou_grad.cu) against the local-frame float64 reference
(oracle.iou_ex_local / iou_ex_grad_local): values and BOTH gradients in fp64 and fp32, far from the origin, on near-collinear and
degenerate pairs, on equivalent parametrisations of a box, over the shapes of the warp-per-box backward and the forward grid, and for
empty, sparse and non-contiguous calls.  Needs a B200: run with `pytest -m gpu`."""
import numpy as np
import pytest
import torch

from conftest import golden, gen_boxes
from iou_ex_cases import (METHODS, OFFSETS, TOL, PINNED_A, PINNED_B, EPS, shifted, collinear_family, turned_family, equivalents,
                          reference, rel_err)

pytestmark = pytest.mark.gpu
SIZES = (1, 7, 8, 9, 31, 32, 33, 257)


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda:0")


def run(a, b, m, up, dev):
    """(value, grad1, grad2) of box2d_iou(a, b, m) in a's dtype (precise=False: fp32 stays fp32) with upstream gradient up"""
    from d3d_b200.box import box2d_iou
    ta = torch.from_numpy(np.ascontiguousarray(a)).to(dev).requires_grad_(True)
    tb = torch.from_numpy(np.ascontiguousarray(b)).to(dev).requires_grad_(True)
    v = box2d_iou(ta, tb, m, precise=False)
    (v * torch.from_numpy(np.ascontiguousarray(up)).to(dev)).sum().backward()
    return v.detach().cpu().numpy(), ta.grad.cpu().numpy(), tb.grad.cpu().numpy()


@pytest.mark.parametrize("dt", [np.float32, np.float64], ids=["f32", "f64"])
def test_translation(dev, oracle, dt):
    """20 x 15 pairs moved by 0 m .. 1 km (fp32) / 100 km (fp64) in a random direction: values and both gradients against the reference.
    "box" and "rbox" values come from iou.cu, "grbox" / "drbox" values and every gradient from iou_grad.cu"""
    vt, gt = TOL[dt]
    worst = {}
    for off in OFFSETS[dt]:
        rng = np.random.default_rng(int(off) + 1)
        a, b = shifted(gen_boxes(rng, 20), gen_boxes(rng, 15), off, rng)
        a, b = a.astype(dt), b.astype(dt)
        up = rng.normal(size=(20, 15)).astype(dt)
        for m in METHODS:
            v, g1, g2, upm, smooth = reference(oracle, a, b, m, up)
            assert smooth.mean() > 0.8, (m, off)
            kv, k1, k2 = run(a, b, m, upm, dev)
            e = (float(np.abs(kv - v).max()), rel_err(k1, g1), rel_err(k2, g2))
            worst[(m, off)] = e
            # iou.cu's "box" forward takes the AABB extents in absolute fp32 coordinates: 2.1e-5 at 1 km (host measurement), inside the
            # 1e-4 IoU bound of fp32 but not the 1e-5 of this file
            v_tol = 1e-4 if (m == "box" and dt == np.float32 and off >= 1e3) else vt
            assert e[0] <= v_tol and e[1] <= gt and e[2] <= gt, (m, off, e)
    print(dt.__name__, {k: "%.1e %.1e %.1e" % e for k, e in worst.items()})


def test_equivalent_boxes(dev):
    """(x, y, w, h, r + pi), (x, y, w, h, r + 2 pi), (x, y, h, w, r + pi / 2): the same rectangle, so the same values and the same
    gradient in x and y, to 1e-12 in fp64"""
    rng = np.random.default_rng(5)
    a, b = gen_boxes(rng, 24) + [0, 0, .3, .3, 0], gen_boxes(rng, 20) + [0, 0, .3, .3, 0]
    up = rng.normal(size=(24, 20))
    for m in ("rbox", "grbox", "drbox"):
        v, g1, g2 = run(a, b, m, up, dev)
        for e in equivalents(b):
            ve, g1e, g2e = run(a, e, m, up, dev)
            assert np.abs(ve - v).max() <= 1e-12 and rel_err(g1e, g1) <= 1e-12 and rel_err(g2e[:, :2], g2[:, :2]) <= 1e-12, m
        for e in equivalents(a):
            ve, g1e, g2e = run(e, b, m, up, dev)
            assert np.abs(ve - v).max() <= 1e-12 and rel_err(g1e[:, :2], g1[:, :2]) <= 1e-12 and rel_err(g2e, g2) <= 1e-12, m


@pytest.mark.parametrize("dt", [np.float32, np.float64], ids=["f32", "f64"])
def test_near_collinear(dev, oracle, dt):
    """B flush with / touching one of A's edges at normal offsets eps (slid along the edge), B turned by a tiny angle about a corner it
    shares with A, and the pinned fp32 pair whose hull was counted twice: values against the reference, continuous in eps"""
    vt = TOL[dt][0]
    rng = np.random.default_rng(21)
    cases = [(PINNED_A.astype(dt), PINNED_B.astype(dt))]
    for off in (0.0, 75.0, 1e3):
        for _ in range(3):
            for a, b in (collinear_family(rng), turned_family(rng)):
                a, b = shifted(a, b, off, rng)
                cases.append((a.astype(dt), b.astype(dt)))
    for a, b in cases:
        for m in ("rbox", "grbox", "drbox"):
            ref = oracle.iou_ex_local(a, b, m)[0]
            got, g1, g2 = run(a, b, m, np.ones((1, len(b)), dt), dev)
            assert np.abs(got[0] - ref).max() <= vt, (m, a, np.abs(got[0] - ref).max())
            assert np.isfinite(g1).all() and np.isfinite(g2).all()
            if len(b) > len(EPS):
                st, sr = np.diff(got[0].reshape(-1, len(EPS)), axis=1), np.diff(ref.reshape(-1, len(EPS)), axis=1)
                assert np.abs(st - sr).max() <= 2 * vt, m
    assert abs(run(PINNED_A, PINNED_B, "grbox", np.ones((1, 1), np.float32), dev)[0][0, 0] - 0.241330) < 1e-5


def test_degenerate_pairs(dev, oracle):
    """The pairs of iou_degenerate.npz (D1-D13: shared corners, flush and coincident edges, headings off by pi / 2 or pi, a zero-width
    box, far apart) and containment / shared-edge pairs: GIoU and DIoU values against the reference in fp64 and fp32, finite gradients.
    Convention for zero-area boxes: with one of them I / U = 0 and the hull / diameter terms follow their definitions; with both the
    union is 0 and the value is 0 (not NaN) for every method."""
    g = golden("iou_degenerate.npz")
    extra_a = np.array([[0, 0, 4, 4, .3], [0, 0, 4, 4, .3], [1, 1, 2, 2, 0], [0, 0, 2, 1, .4], [3, -1, 2, 2, 0]])
    extra_b = np.array([[.5, -.2, 1, 2, 1.1],                                # B inside A
                        [0, 0, 4, 4, .3 + np.pi / 2],                        # identical square, other parametrisation
                        [3, 1, 2, 2, 0],                                     # shared edge, opposite sides
                        [0, 0.75, 2, .5, .4],                                # inside, flush with A's top edge (rotated)
                        [4, -1, 2, 2, 0]])                                   # overlap, collinear top and bottom edges
    a_all, b_all = np.concatenate([g["boxes1"], extra_a]), np.concatenate([g["boxes2"], extra_b])
    for dt, vt in ((np.float64, 1e-10), (np.float32, 1e-5)):
        a_, b_ = a_all.astype(dt), b_all.astype(dt)
        for m in ("rbox", "grbox", "drbox"):
            for i in range(len(a_)):
                ref = oracle.iou_ex_local(a_[i:i + 1], b_[i:i + 1], m)[0, 0]
                v, g1, g2 = run(a_[i:i + 1], b_[i:i + 1], m, np.ones((1, 1), dt), dev)
                assert abs(v[0, 0] - ref) <= vt, (m, dt.__name__, i, v[0, 0], ref)
                assert np.isfinite(g1).all() and np.isfinite(g2).all(), (m, i)
    z, z2 = np.array([[0, 0, 0, 2, .2]]), np.array([[5, 5, 0, 0, .1]])
    for m in METHODS:
        v, g1, g2 = run(z, z2, m, np.ones((1, 1)), dev)
        assert v[0, 0] == 0.0 and np.isfinite(g1).all() and np.isfinite(g2).all(), m


@pytest.mark.parametrize("m", ["grbox", "drbox", "rbox", "box"])
def test_backward_shapes(dev, oracle, m):
    """(n, m) over 1, 7, 8, 9, 31, 32, 33, 257 on both sides (one warp per owned box, 8 per CTA, the other side strided by 32 lanes):
    small shapes against the reference, every shape against the sum of the same backward over column (grad1) and row (grad2) chunks"""
    rng = np.random.default_rng(17)
    for n in SIZES:
        for k in SIZES:
            a, b = gen_boxes(rng, n), gen_boxes(rng, k)
            up = rng.normal(size=(n, k))
            if n * k <= 64:
                rv, rg1, rg2, up, _ = reference(oracle, a, b, m, up)
            v, g1, g2 = run(a, b, m, up, dev)
            if n * k <= 64:
                assert np.abs(v - rv).max() <= 1e-10 and rel_err(g1, rg1) <= 1e-8 and rel_err(g2, rg2) <= 1e-8, (m, n, k)
            s1 = sum(run(a, b[c:c + 13], m, up[:, c:c + 13], dev)[1] for c in range(0, k, 13))
            s2 = sum(run(a[r:r + 13], b, m, up[r:r + 13], dev)[2] for r in range(0, n, 13))
            assert rel_err(g1, s1) <= 1e-12 and rel_err(g2, s2) <= 1e-12, (m, n, k)


@pytest.mark.parametrize("dt", [np.float32, np.float64], ids=["f32", "f64"])
def test_forward_grid(dev, oracle, dt):
    """GIoU / DIoU forward: one 256-thread CTA per 256 columns, one grid row per box row, launched in chunks of 65535 rows"""
    from d3d_b200.box import box2d_iou
    vt = TOL[dt][0]
    rng = np.random.default_rng(29)
    for k in (1, 255, 256, 257):
        a, b = gen_boxes(rng, 3).astype(dt), gen_boxes(rng, k).astype(dt)
        for m in ("grbox", "drbox"):
            v = box2d_iou(torch.from_numpy(a).to(dev), torch.from_numpy(b).to(dev), m, precise=False).cpu().numpy()
            assert v.shape == (3, k) and np.abs(v - oracle.iou_ex_local(a, b, m)).max() <= vt, (m, k)
    a, b = gen_boxes(rng, 65537, spread=40.0).astype(dt), gen_boxes(rng, 3).astype(dt)
    rows = np.r_[0:3, 65530:65537]
    for m in ("grbox", "drbox"):
        v = box2d_iou(torch.from_numpy(a).to(dev), torch.from_numpy(b).to(dev), m, precise=False).cpu().numpy()
        assert v.shape == (65537, 3) and np.isfinite(v).all(), m
        assert np.abs(v[rows] - oracle.iou_ex_local(a[rows], b, m)).max() <= vt, m


def test_calls(dev, oracle):
    """an empty side (the backward memsets: exact zeros), a sparse upstream gradient (the up == 0 skip), a non-contiguous one"""
    from d3d_b200.box import box2d_iou
    rng = np.random.default_rng(33)
    a, b = gen_boxes(rng, 5), gen_boxes(rng, 5)
    for m in METHODS:
        for x, y in ((a, np.zeros((0, 5))), (np.zeros((0, 5)), b)):
            tx, ty = (torch.from_numpy(t).to(dev).requires_grad_(True) for t in (x, y))
            v = box2d_iou(tx, ty, m)
            assert v.shape == (len(x), len(y))
            v.sum().backward()
            assert torch.equal(tx.grad, torch.zeros_like(tx)) and torch.equal(ty.grad, torch.zeros_like(ty)), m
    a, b = gen_boxes(rng, 20), gen_boxes(rng, 15)
    up = np.zeros(300)
    up[rng.choice(300, 24, replace=False)] = rng.normal(size=24)   # 24 of 300 non-zero: 92 % exact zeros
    up = up.reshape(20, 15)
    assert (up == 0).mean() >= 0.9
    for m in METHODS:
        rv, rg1, rg2, upm, _ = reference(oracle, a, b, m, up)
        v, g1, g2 = run(a, b, m, upm, dev)
        assert rel_err(g1, rg1) <= 1e-8 and rel_err(g2, rg2) <= 1e-8, m
        ta, tb = (torch.from_numpy(t).to(dev).requires_grad_(True) for t in (a, b))
        w = torch.from_numpy(np.ascontiguousarray(upm.T)).to(dev)
        (box2d_iou(ta, tb, m).t() * w).sum().backward()   # the upstream gradient reaches the backward as a transposed view
        assert torch.equal(ta.grad.cpu(), torch.from_numpy(g1)) and torch.equal(tb.grad.cpu(), torch.from_numpy(g2)), m
