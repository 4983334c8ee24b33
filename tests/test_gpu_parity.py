"""Parity tests proper: the CUDA path (through the Python front doors -> C ABI -> kernels) against the
CPU oracle and the committed golden fixtures, plus size-independent properties at BASELINE sizes.
Needs a B200: run with `pytest -m gpu`."""
import numpy as np
import pytest
import torch

from conftest import golden, gen_boxes, lidar, proposals, SOFT_CASES, SOFT_TEST6, soft_inputs
from d3d_b200 import _cabi

pytestmark = pytest.mark.gpu

FP64_TOL = 1e-5   # north_star: IoU within 1e-5 absolute in fp64
FP32_TOL = 1e-4   # and 1e-4 in fp32


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda:0")


def _unpack(bits, n):
    return np.unpackbits(bits)[:n].astype(bool)


def _t(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


# ------------------------------------------------------------------ IoU
def test_iou_golden_reference_fixture(dev):
    from d3d_b200.box import box2d_iou
    g = golden("iou_c1.npz")
    a, b = g["boxes1"], g["boxes2"]
    r = box2d_iou(_t(a, dev), _t(b, dev), "rbox").cpu().numpy()
    assert r.dtype == np.float64 and np.abs(r - g["rbox_f64"]).max() < FP64_TOL
    assert np.abs(r - g["rbox_f64"]).max() < 1e-10   # in generic position we are ~1e-13 from the reference
    r = box2d_iou(_t(a, dev), _t(b, dev), "box").cpu().numpy()
    assert np.abs(r - g["box_f64"]).max() < 1e-12
    a32, b32 = a.astype(np.float32), b.astype(np.float32)
    r32 = box2d_iou(_t(a32, dev), _t(b32, dev), "rbox", precise=False).cpu().numpy()
    assert r32.dtype == np.float32 and np.abs(r32 - g["rbox_f32"]).max() < FP32_TOL
    assert np.abs(box2d_iou(_t(a32, dev), _t(b32, dev), "box", precise=False).cpu().numpy() - g["box_f32"]).max() < 1e-5
    # precise=True on float input: fp64 compute, float result (d3d/box/__init__.py:197-221)
    rp = box2d_iou(_t(a32, dev), _t(b32, dev), "rbox")
    assert rp.dtype == torch.float32


def test_iou_c1_full_vs_oracle(dev, oracle):
    """config C1: 1k x 1k fp64 + fp32 against the oracle (reference RC restatement) and truth."""
    from d3d_b200.box import box2d_iou
    rng = np.random.default_rng(0)
    A, B = gen_boxes(rng, 1000), gen_boxes(rng, 1000)
    r = box2d_iou(_t(A, dev), _t(B, dev), "rbox").cpu().numpy()
    ref = oracle.iou2dr(A, B)
    assert np.abs(r - ref).max() < 1e-10
    assert abs(r.sum() - 20745.014676358896) < 1e-6 and (r != 0).sum() == 205623   # SURVEY Appendix C anchors
    A32, B32 = A.astype(np.float32), B.astype(np.float32)
    r32 = box2d_iou(_t(A32, dev), _t(B32, dev), "rbox", precise=False).cpu().numpy()
    truth = oracle.iou2dr_truth(A32.astype(np.float64), B32.astype(np.float64))
    assert np.abs(r32 - truth).max() < 2e-6
    assert np.abs(r32 - oracle.iou2dr(A32, B32)).max() < FP32_TOL
    rb = box2d_iou(_t(A, dev), _t(B, dev), "box").cpu().numpy()
    assert np.abs(rb - oracle.iou2d(A, B)).max() < 1e-12


def test_iou_reference_known_answers(dev):
    """test/test_box.py:12-100 with the reference's tolerances, CUDA and host inputs, numpy round trip."""
    from d3d_b200.box import box2d_iou
    g = golden("iou_known_answers.npz")
    eps = 1e-3
    for mv in (lambda x: _t(x, dev), lambda x: torch.from_numpy(x), lambda x: x):
        def run(a, b, m):
            r = box2d_iou(mv(a), mv(b), method=m)
            return r if isinstance(r, np.ndarray) else r.cpu().numpy()
        assert np.allclose(run(g["aa_boxes1"], g["aa_boxes2"], "box"), g["aa_expected"], atol=eps)
        assert np.allclose(run(g["aa_boxes1"], g["aa_boxes2"], "rbox"), g["aa_expected"], atol=4 * eps)
        assert np.allclose(run(g["rot_boxes1"], g["rot_boxes2"], "box"), g["rot_box_expected"], atol=2 * eps)
        assert np.allclose(run(g["rot_boxes1"], g["rot_boxes2"], "rbox"), g["rot_rbox_expected"], atol=4 * eps)
        ab = g["apart_boxes"]
        assert np.allclose(run(ab, ab, "box") - np.eye(4), 0, atol=1e-6)
        rb = g["apart_rboxes"]
        assert np.allclose(run(rb, rb, "rbox") - np.eye(5), 0, atol=1e-6)


def test_iou_degenerate_list(dev):
    """SURVEY 8(c) D1-D13: the build returns geometric truth where the reference's RC returns 1.0/0.5."""
    from d3d_b200.box import box2d_iou
    g = golden("iou_degenerate.npz")
    for i, name in enumerate(g["names"]):
        a, b = g["boxes1"][i:i + 1], g["boxes2"][i:i + 1]
        v64 = box2d_iou(_t(a, dev), _t(b, dev), "rbox").item()
        v32 = box2d_iou(_t(a.astype(np.float32), dev), _t(b.astype(np.float32), dev), "rbox", precise=False).item()
        assert abs(v64 - g["truth"][i]) < FP64_TOL, (name, v64)
        assert abs(v32 - g["truth"][i]) < FP32_TOL, (name, v32)
        if str(name) == "D13":
            assert v64 == 0.0 and v32 == 0.0 and not np.signbit(v64)   # early reject yields exactly +0
    z = np.array([[0, 0, 0, 2, .2]]); z2 = np.array([[5, 5, 0, 0, .1]])
    assert box2d_iou(_t(z, dev), _t(z2, dev), "rbox").item() == 0.0   # two zero-area boxes: 0, not NaN (documented)


def test_iou_shapes_edges_and_errors(dev, oracle):
    from d3d_b200.box import box2d_iou
    rng = np.random.default_rng(3)
    for n, m in ((1, 1), (1, 257), (63, 129), (65, 127), (200, 3), (130, 1001)):   # ragged tiles, unaligned ld
        A, B = gen_boxes(rng, n), gen_boxes(rng, m)
        for dt, tol in ((np.float64, 1e-10), (np.float32, FP32_TOL)):
            r = box2d_iou(_t(A.astype(dt), dev), _t(B.astype(dt), dev), "rbox", precise=False).cpu().numpy()
            assert r.shape == (n, m) and np.abs(r - oracle.iou2dr(A.astype(dt), B.astype(dt))).max() < tol
            rb = box2d_iou(_t(A.astype(dt), dev), _t(B.astype(dt), dev), "box", precise=False).cpu().numpy()
            assert np.abs(rb - oracle.iou2d(A.astype(dt), B.astype(dt))).max() < (1e-12 if dt == np.float64 else 1e-5)
    e = box2d_iou(torch.zeros((0, 5), device=dev), torch.zeros((7, 5), device=dev), "rbox")
    assert e.shape == (0, 7)
    with pytest.raises(ValueError):
        box2d_iou(torch.zeros((3, 4), device=dev), torch.zeros((3, 5), device=dev), "rbox")
    with pytest.raises(ValueError):
        box2d_iou(torch.zeros(5, device=dev), torch.zeros((3, 5), device=dev))
    with pytest.raises(AttributeError):
        box2d_iou(torch.zeros((3, 5), device=dev), torch.zeros((3, 5), device=dev), "nonsense")
    # non-contiguous inputs are accepted like the reference's strided accessors
    big = _t(gen_boxes(rng, 40), dev)
    assert torch.equal(box2d_iou(big[::2], big[1::2], "rbox"), box2d_iou(big[::2].contiguous(), big[1::2].contiguous(), "rbox"))


def test_iou_large_properties(dev, oracle):
    """20k x 20k fp32 (4e8 pairs): range, symmetry, diagonal, sampled rows vs truth; test_box.py:125-138."""
    from d3d_b200.box import box2d_iou
    rng = np.random.default_rng(9)
    n = 20000
    A = gen_boxes(rng, n, spread=60.0).astype(np.float32)
    tA = _t(A, dev)
    r = box2d_iou(tA, tA, "rbox", precise=False)
    assert r.shape == (n, n) and bool(((r >= -1e-3) & (r <= 1 + 1e-3)).all())
    assert float((r - r.t()).abs().max()) < FP32_TOL
    assert float((torch.diagonal(r) - 1).abs().max()) < FP32_TOL
    rows = rng.integers(0, n, 24)
    truth = oracle.iou2dr_truth(A[rows].astype(np.float64), A.astype(np.float64))
    assert np.abs(r[torch.from_numpy(rows).to(dev)].cpu().numpy() - truth).max() < FP32_TOL
    x = torch.rand(500) * 200; y = torch.rand(500) * 400
    b = torch.stack((x, y, torch.rand(500) * 20 + 10, torch.rand(500) * 30 + 5, torch.rand(500) * 2 - 1), dim=1).to(dev)
    for m in ("box", "rbox"):
        res = box2d_iou(b, b, method=m)
        assert bool(torch.all(res >= -1e-3)) and bool(torch.all(res <= 1 + 1e-3))


# ------------------------------------------------------------------ NMS
def _boxes3d(rng, n, extent=40.0):
    return np.stack([(rng.random(n) - .5) * extent, (rng.random(n) - .5) * extent, rng.normal(-1, 0.5, n),
                     3.5 + rng.random(n) * 2, 1.5 + rng.random(n), 1.4 + rng.random(n) * 0.6, (rng.random(n) - .5) * 7], 1).astype(np.float32)


def test_iou_differentiable_family(dev, oracle):
    """A2 / f2: box2d_iou is differentiable for its four methods.  Values of GIoU / DIoU and all gradients against the fixture written by
    the reference's own forward / backward (fp64, single-threaded), torch.autograd.gradcheck on generic pairs, the fp32 path against
    the fp64 one, identical boxes, numpy and host inputs."""
    from d3d_b200.box import box2d_iou, Iou2DR, GIou2DR
    g = golden("iou_grad.npz")
    A, B, up = g["boxes1"], g["boxes2"], g["grad"]
    for m, vtol in (("box", 1e-12), ("rbox", 1e-10), ("grbox", 1e-10), ("drbox", 1e-10)):
        a, b = _t(A, dev).requires_grad_(True), _t(B, dev).requires_grad_(True)
        v = box2d_iou(a, b, m)
        assert v.requires_grad and np.abs(v.detach().cpu().numpy() - g[m + ".value"]).max() < vtol, m
        (v * _t(up, dev)).sum().backward()
        assert np.abs(a.grad.cpu().numpy() - g[m + ".grad1"]).max() < 1e-8, (m, float(np.abs(a.grad.cpu().numpy() - g[m + ".grad1"]).max()))
        assert np.abs(b.grad.cpu().numpy() - g[m + ".grad2"]).max() < 1e-8, (m, float(np.abs(b.grad.cpu().numpy() - g[m + ".grad2"]).max()))
        a32, b32 = _t(A.astype(np.float32), dev).requires_grad_(True), _t(B.astype(np.float32), dev).requires_grad_(True)
        v32 = box2d_iou(a32, b32, m, precise=False)
        assert v32.dtype == torch.float32 and np.abs(v32.detach().cpu().numpy() - g[m + ".value"]).max() < FP32_TOL
        (v32 * _t(up.astype(np.float32), dev)).sum().backward()
        assert np.abs(a32.grad.cpu().numpy() - g[m + ".grad1"]).max() < 5e-3 * max(1.0, np.abs(g[m + ".grad1"]).max())
    rng = np.random.default_rng(5)
    a = _t(gen_boxes(rng, 5, spread=4.0) + np.array([0, 0, .5, .5, 0]), dev).requires_grad_(True)
    b = _t(gen_boxes(rng, 4, spread=4.0) + np.array([0, 0, .5, .5, 0]), dev).requires_grad_(True)
    for m in ("box", "rbox", "grbox", "drbox"):
        assert torch.autograd.gradcheck(lambda x, y: box2d_iou(x, y, m), (a, b), eps=1e-6, atol=1e-5, rtol=1e-4, nondet_tol=0.0), m
    same = _t(A[:8], dev)
    assert np.abs(box2d_iou(same, same, "grbox").diagonal().cpu().numpy() - 1).max() < 1e-12      # identical boxes: shared edges counted once
    assert np.abs(box2d_iou(same, same, "drbox").diagonal().cpu().numpy() - 1).max() < 1e-12
    assert np.abs(box2d_iou(A, B, "grbox") - g["grbox.value"]).max() < 1e-10                       # numpy in, numpy out
    hv = box2d_iou(torch.from_numpy(A).requires_grad_(True), torch.from_numpy(B), "drbox")         # host tensors: differentiable through the copies
    hv.sum().backward()
    assert not hv.is_cuda
    far = _t(A[:3] + np.array([1000, 0, 0, 0, 0]), dev).requires_grad_(True)                       # no overlap: zero IoU gradient, non-zero GIoU gradient
    box2d_iou(far, _t(B, dev), "rbox").sum().backward()
    assert float(far.grad.abs().max()) == 0.0
    far.grad = None
    box2d_iou(far, _t(B, dev), "grbox").sum().backward()
    assert float(far.grad.abs().max()) > 0.0
    assert Iou2DR.__name__ == "Iou2DR" and issubclass(GIou2DR, torch.autograd.Function)


def test_box3d_iou_distance_vs_oracle(dev, oracle):
    """SURVEY 8(f) row f1: the evaluator's distance matrix 1 - iou2d * ziou (fp32).  Against geometric truth everywhere
    (tolerance 1e-4, north_star's fp32 bound), against the reference's own fp32 Rotating-Calipers path on the pairs where
    that path is sane, and bit-exact for the axis-aligned metric, whose arithmetic has no transcendental in the pair loop."""
    from d3d_b200.box import box3d_iou_distance
    rng = np.random.default_rng(31)
    for n, m in ((1, 1), (37, 129), (300, 257), (1000, 700)):
        A, B = _boxes3d(rng, n), _boxes3d(rng, m)
        B[: min(n, m) // 3] = A[: min(n, m) // 3] + rng.normal(0, 0.15, (min(n, m) // 3, 7)).astype(np.float32)   # true matches
        d = box3d_iou_distance(_t(A, dev), _t(B, dev), "riou")
        assert d.dtype == torch.float32 and tuple(d.shape) == (n, m)
        d = d.cpu().numpy()
        truth = oracle.box3d_iou_distance(A, B, "riou", alg=oracle.ALG_TRUTH)
        assert np.abs(d - truth).max() < 1e-4, (n, m, float(np.abs(d - truth).max()))
        ref = oracle.box3d_iou_distance(A, B, "riou")
        sane = np.abs(ref - truth) < 1e-4                                    # the fp32 RC path blows up on rare pairs (SURVEY 8(c))
        assert sane.mean() > 0.999 and np.abs(d - ref)[sane].max() < 2e-4
        assert d.min() >= -1e-6 and d.max() <= 1.0 + 1e-6
        da = box3d_iou_distance(_t(A, dev), _t(B, dev), "iou").cpu().numpy()
        assert np.abs(da - oracle.box3d_iou_distance(A, B, "iou")).max() < 2e-6
    # z semantics: identical boxes -> 0, disjoint in z -> 1, half z overlap of the same footprint -> 1 - 1/3, flat boxes (u clamp)
    a = np.array([[0, 0, 0, 4, 2, 2, 0.3]], np.float32)
    cases = np.array([[0, 0, 0, 4, 2, 2, 0.3], [0, 0, 5, 4, 2, 2, 0.3], [0, 0, 1, 4, 2, 2, 0.3], [0, 0, 0, 4, 2, 0, 0.3]], np.float32)
    got = box3d_iou_distance(a, cases, "riou")
    assert isinstance(got, np.ndarray) and np.allclose(got[0], [0.0, 1.0, 1 - 1 / 3, 1.0], atol=2e-6)
    flat = np.array([[0, 0, 0, 4, 2, 0, 0.3]], np.float32)
    assert np.allclose(box3d_iou_distance(flat, flat, "riou"), oracle.box3d_iou_distance(flat, flat, "riou", alg=oracle.ALG_TRUTH), atol=1e-6)
    assert box3d_iou_distance(torch.zeros((0, 7)), torch.zeros((5, 7))).shape == (0, 5)
    g = golden("dist3d.npz")   # written by the reference's own box3dr_iou / box3d_iou (d3d/dgal_wrap.h, g++)
    truth = oracle.box3d_iou_distance(g["src"], g["dst"], "riou", alg=oracle.ALG_TRUTH)
    sane = np.abs(g["riou"] - truth) < 1e-4
    assert np.abs(box3d_iou_distance(g["src"], g["dst"], "riou") - g["riou"])[sane].max() < 2e-4
    assert np.abs(box3d_iou_distance(g["src"], g["dst"], "iou") - g["iou"]).max() < 2e-6
    with pytest.raises(ValueError):
        box3d_iou_distance(torch.zeros((3, 5)), torch.zeros((3, 7)))
    with pytest.raises(ValueError):
        box3d_iou_distance(torch.zeros((3, 7)), torch.zeros((3, 7)), metric="giou")


def test_match_greedy_vs_oracle(dev, oracle):
    """f1: greedy score-ordered matching of the detection evaluator (ScoreMatcher.match), 40 threshold sets in one launch, against the
    restated walk; distances come from the distance-matrix kernel, so the pipeline prepare_boxes -> match runs on the device"""
    from d3d_b200.box import box3d_iou_distance, match_greedy
    rng = np.random.default_rng(41)
    for n, m, ncat in ((1, 1, 1), (60, 45, 3), (400, 350, 4)):
        A, B = _boxes3d(rng, n), _boxes3d(rng, m)
        k = min(n, m) // 2
        B[:k] = A[:k] + rng.normal(0, 0.2, (k, 7)).astype(np.float32)
        st, dt = rng.integers(0, ncat, n), rng.integers(0, ncat, m)
        dt[:k] = st[:k]
        scores = rng.random(n)
        d = box3d_iou_distance(_t(A, dev), _t(B, dev), "riou")
        thr = np.stack([np.full(ncat, 1 - t) + rng.random(ncat) * 0.05 for t in np.linspace(0.1, 0.9, 40)]).astype(np.float32)
        sa, da = match_greedy(d, _t(scores, dev), _t(st, dev), _t(dt, dev), _t(thr, dev))
        assert sa.shape == (40, n) and da.shape == (40, m) and sa.dtype == torch.int32
        dn = d.cpu().numpy()
        for t in (0, 13, 39):
            osa, oda = oracle.match_greedy(dn, scores, st, dt, thr[t])
            assert np.array_equal(sa[t].cpu().numpy(), osa) and np.array_equal(da[t].cpu().numpy(), oda), (n, m, t)
        s1, d1 = match_greedy(dn, scores, st, dt, thr[5])          # numpy in, numpy out, single threshold set
        assert isinstance(s1, np.ndarray) and np.array_equal(s1, oracle.match_greedy(dn, scores, st, dt, thr[5])[0])
    sa, da = match_greedy(torch.zeros((0, 4)), [], [], [0, 0, 0, 0], [0.5])
    assert sa.shape == (0,) and da.tolist() == [-1, -1, -1, -1]


def test_box_crop_vs_reference_and_oracle(dev, oracle):
    """SURVEY 8(f) row f4: box2dr_crop / box3dp_crop.  Masks are compared bit for bit with the golden fixture written by the
    reference's own crop_2dr and with the oracle on ragged sizes; points closer than a few ulps to an edge could flip with
    the last-ulp difference between CUDA's and glibc's sin/cos (none do on these inputs)."""
    from d3d_b200.box import box2dr_crop, box3dp_crop
    g = golden("crop.npz")
    for tag in ("f32", "f64"):
        pts, bx = g[f"{tag}.points"], g[f"{tag}.boxes"]
        exp = np.unpackbits(g[f"{tag}.mask"])[:len(bx) * len(pts)].reshape(len(bx), len(pts)).astype(bool)
        got = box2dr_crop(_t(pts, dev), _t(bx, dev))
        assert got.dtype == torch.bool and tuple(got.shape) == exp.shape
        assert np.array_equal(got.cpu().numpy(), exp), (tag, int((got.cpu().numpy() != exp).sum()))
    rng = np.random.default_rng(17)
    for n, m in ((1, 1), (15, 3), (16, 17), (4099, 33), (70000, 40), (65536, 16)):
        for dt in (np.float32, np.float64):
            pts = ((rng.random((n, 2)) - .5) * 12).astype(dt)
            bx = gen_boxes(rng, m).astype(dt)
            exp = oracle.crop_2dr(pts, bx)
            for path in ("brute", "grid"):   # both back ends (the grid over the points is the default from 64 M pairs on)
                _cabi.tuning_set("D3D_B200_CROP_PATH", {"brute": 1, "grid": 2}[path])
                got = box2dr_crop(_t(pts, dev), _t(bx, dev)).cpu().numpy()
                assert np.array_equal(got, exp), (n, m, dt, path)
            _cabi.tuning_set("D3D_B200_CROP_PATH", None)
    # grid path corner cases: boxes far outside the cloud, a degenerate (flat) box, clustered points, a NaN point (falls back to brute force)
    pts = np.concatenate([rng.normal(0, 0.01, (5000, 2)), (rng.random((5000, 2)) - .5) * 200]).astype(np.float32)
    bx = np.array([[0, 0, 0.05, 0.05, 0.4], [1e6, 1e6, 5, 5, 0], [0, 0, 0, 3, 1], [0, 0, 400, 400, 0.1], [-90, 95, 30, 2, 2.0]], np.float32)
    _cabi.tuning_set("D3D_B200_CROP_PATH", 2)
    assert np.array_equal(box2dr_crop(_t(pts, dev), _t(bx, dev)).cpu().numpy(), oracle.crop_2dr(pts, bx))
    pts[17] = np.nan
    assert np.array_equal(box2dr_crop(_t(pts, dev), _t(bx, dev)).cpu().numpy(), oracle.crop_2dr(pts, bx))
    one = np.zeros((300, 2), np.float32)
    assert np.array_equal(box2dr_crop(_t(one, dev), _t(bx, dev)).cpu().numpy(), oracle.crop_2dr(one, bx))
    _cabi.tuning_set("D3D_B200_CROP_PATH", None)
    # bench size (180k lidar-like points x 4096 proposals: boxes on the dense first metres have tens of thousands of candidates):
    # the grid path against the brute-force path over the whole mask, and against the oracle on sampled rows
    from bench import lidar as bench_lidar, proposals as bench_proposals
    pts = bench_lidar(300, 180_000)[:, :2].copy()
    bx = bench_proposals(300, 4096, 2048)[0].astype(np.float32)
    tp, tb = _t(pts, dev), _t(bx, dev)
    _cabi.tuning_set("D3D_B200_CROP_PATH", 1)
    brute = box2dr_crop(tp, tb)
    _cabi.tuning_set("D3D_B200_CROP_PATH", 2)
    grid = box2dr_crop(tp, tb)
    _cabi.tuning_set("D3D_B200_CROP_PATH", None)
    assert torch.equal(brute, grid) and int(grid.sum()) > 0
    rows = rng.integers(0, 4096, 24)
    assert np.array_equal(grid[torch.from_numpy(rows).to(dev)].cpu().numpy(), oracle.crop_2dr(pts, bx[rows]))
    # reference test/test_box.py:191-205
    cloud = (rng.random((100, 2)) * 2 - 1).astype(np.float32)
    boxes = np.array([[0, 0, 1, 1, 0], [0, 0, 1, 1, np.pi / 4]], np.float32)
    r = box2dr_crop(torch.from_numpy(cloud), torch.from_numpy(boxes))
    assert r.device.type == "cpu"
    ab = np.abs(cloud)
    assert np.array_equal(r[0].numpy(), np.all(ab < 0.5, 1)) and np.array_equal(r[1].numpy(), np.abs(ab[:, 0] + ab[:, 1]) < np.sqrt(2) / 2)
    p3 = np.concatenate([(rng.random((5000, 2)) - .5) * 12, rng.normal(0, 1, (5000, 1))], 1).astype(np.float32)
    b3 = np.concatenate([gen_boxes(rng, 20)[:, :2], rng.normal(0, .5, (20, 1)), gen_boxes(rng, 20)[:, 2:4], 1 + rng.random((20, 1)), rng.normal(0, 2, (20, 1))], 1).astype(np.float32)
    for ax in (0, 1, 2):
        assert np.array_equal(box3dp_crop(_t(p3, dev), _t(b3, dev), ax).cpu().numpy(), oracle.box3dp_crop(p3, b3, ax)), ax
    assert tuple(box2dr_crop(torch.zeros((0, 2), device=dev), torch.zeros((4, 5), device=dev)).shape) == (4, 0)
    with pytest.raises(ValueError):
        box2dr_crop(torch.zeros((3, 3), device=dev), torch.zeros((4, 5), device=dev))
    with pytest.raises(ValueError):
        box3dp_crop(_t(p3, dev), _t(b3, dev), 3)


def test_nms_known_answer_and_golden(dev):
    from d3d_b200.box import box2d_nms
    g = golden("nms.npz")
    for m in ("box", "rbox"):
        k = box2d_nms(_t(g["test_boxes"], dev), _t(g["test_scores"], dev), iou_method=m)
        assert k.dtype == torch.bool and np.array_equal(k.cpu().numpy(), g["test_expected"])
    A, B, s = g["c1_boxes"], g["c1_boxes_b"], g["c1_scores"]
    k = box2d_nms(_t(A, dev), _t(s, dev), "rbox", iou_threshold=0.5).cpu().numpy()
    assert k.sum() == 673 and np.array_equal(k, _unpack(g["c1_keep_rbox"], 1000))
    assert np.array_equal(box2d_nms(_t(B, dev), _t(s, dev), "rbox", iou_threshold=0.5).cpu().numpy(), _unpack(g["c1_keep_rbox_b"], 1000))
    assert np.array_equal(box2d_nms(_t(A, dev), _t(s, dev), "box", iou_threshold=0.5).cpu().numpy(), _unpack(g["c1_keep_box"], 1000))
    assert np.array_equal(box2d_nms(_t(A, dev), _t(s, dev), "rbox", iou_threshold=0.3, score_threshold=0.2).cpu().numpy(),
                          _unpack(g["c1_keep_rbox_thr03_s02"], 1000))
    P, ps = g["prop_boxes"], g["prop_scores"]
    assert np.array_equal(box2d_nms(_t(P, dev), _t(ps, dev), "rbox", iou_threshold=0.5).cpu().numpy(), _unpack(g["prop_keep_rbox"], len(P)))
    assert np.array_equal(box2d_nms(_t(P, dev), _t(ps, dev), "box", iou_threshold=0.5).cpu().numpy(), _unpack(g["prop_keep_box"], len(P)))
    # numpy in -> numpy out; host tensors in -> host tensors out
    kn = box2d_nms(A, s, "rbox", iou_threshold=0.5)
    assert isinstance(kn, np.ndarray) and np.array_equal(kn, _unpack(g["c1_keep_rbox"], 1000))
    # fp32 path (precise=False): near-threshold pairs are re-evaluated in fp64, so the float32 keep mask of
    # float32-rounded boxes equals the reference's fp64 decisions on those same boxes
    P32, ps32 = P.astype(np.float32), ps.astype(np.float32)
    if len(np.unique(ps32)) == len(ps32):
        k32 = box2d_nms(_t(P32, dev), _t(ps32, dev), "rbox", iou_threshold=0.5, precise=False).cpu().numpy()
        assert np.array_equal(k32, box2d_nms(_t(P32, dev), _t(ps32, dev), "rbox", iou_threshold=0.5, precise=True).cpu().numpy())


def test_nms_vs_oracle_sizes_and_thresholds(dev, oracle):
    from d3d_b200.box import box2d_nms
    rng = np.random.default_rng(21)
    for n in (1, 2, 63, 64, 65, 130, 1000, 4097):
        P, s = proposals(rng, n, max(1, n // 25), extent=20.0)
        for m in ("rbox", "box"):
            for thr, sthr in ((0.5, 0.0), (0.3, 0.35), (0.0, 0.0), (0.7, 0.999)):
                k = box2d_nms(_t(P, dev), _t(s, dev), m, iou_threshold=thr, score_threshold=sthr).cpu().numpy()
                o = oracle.box2d_nms(P, s, m, iou_threshold=thr, score_threshold=sthr, cuda_score_rule=True)
                assert np.array_equal(k, o), (n, m, thr, sthr, int((k != o).sum()))
                assert not k[s <= sthr].any()          # test_box.py:140-155
                if s.max() > sthr:                      # the CPU rule only differs when every score is <= thr (T4)
                    assert np.array_equal(k, oracle.box2d_nms(P, s, m, iou_threshold=thr, score_threshold=sthr))
    assert box2d_nms(torch.zeros((0, 5), device=dev), torch.zeros(0, device=dev)).numel() == 0
    with pytest.raises(ValueError):
        box2d_nms(torch.zeros((3, 5), device=dev), torch.zeros(2, device=dev))
    with pytest.raises(AttributeError):   # reference: getattr(SupressionType, "SOFT") fails the same way
        box2d_nms(torch.rand((3, 5), device=dev), torch.rand(3, device=dev), supression_method="soft")
    # 2-D scores: max over classes (d3d/box/__init__.py:253-254)
    P, s = proposals(rng, 300, 12, extent=10.0)
    s2 = np.stack([s * 0.5, s, s * 0.1], 1)
    assert np.array_equal(box2d_nms(_t(P, dev), _t(s2, dev), "rbox", iou_threshold=0.4).cpu().numpy(),
                          oracle.box2d_nms(P, s, "rbox", iou_threshold=0.4, cuda_score_rule=True))


def test_nms_soft_vs_reference_and_oracle(dev, oracle):
    """f3: LINEAR / GAUSSIAN suppression.  Keep masks equal, bit for bit in fp64, to the fixtures written by the reference's own CPU
    nms2d (n = 6, 1000, 4097) and to the oracle on fresh inputs; the fp32 path agrees with the fp64 one up to near-threshold pairs."""
    from d3d_b200.box import box2d_nms
    g = golden("nms_soft.npz")
    nb, ns = SOFT_TEST6
    for m, par in (("linear", 1.0), ("gaussian", 0.5)):
        for im in ("box", "rbox"):
            keep = box2d_nms(_t(nb, dev), _t(ns, dev), im, m, iou_threshold=0.1, score_threshold=0.15, supression_param=par)
            assert keep.dtype == torch.bool and np.array_equal(keep.cpu().numpy(), g[f"test6_{m}_{im}"]), (m, im)
    for tag, n, gen, m, it, st, par in SOFT_CASES:
        b, s = soft_inputs(n, gen)
        im = "box" if tag.endswith("_box") else "rbox"
        keep = box2d_nms(_t(b, dev), _t(s, dev), im, m, iou_threshold=it, score_threshold=st, supression_param=par).cpu().numpy()
        exp = _unpack(g[tag], n)
        assert np.array_equal(keep, exp), (tag, int((keep != exp).sum()))
        k32 = box2d_nms(_t(b.astype(np.float32), dev), _t(s.astype(np.float32), dev), im, m, iou_threshold=it, score_threshold=st,
                        supression_param=par, precise=False).cpu().numpy()
        assert (k32 != exp).mean() < 0.02, (tag, "fp32", int((k32 != exp).sum()))
    rng = np.random.default_rng(77)
    for n in (1, 2, 65, 300):
        b, s = gen_boxes(rng, n, spread=4.0), rng.random(n)
        for m, par in (("linear", 0.7), ("gaussian", 0.4)):
            keep = box2d_nms(b, s, "rbox", m, iou_threshold=0.2, score_threshold=0.25, supression_param=par)   # numpy in, numpy out
            assert np.array_equal(keep, oracle.box2d_nms(b, s, "rbox", m, 0.2, 0.25, par, cuda_score_rule=True)), (n, m)


def test_nms_batch_equals_per_frame(dev, oracle):
    """J1 (BASELINE.json config 5): frame-batched hard NMS == one box2d_nms call per frame == oracle, for ragged frames (empty, one box,
    exactly 64, 4096 proposals), both IoU methods, fp64 and fp32, list and packed call forms"""
    from d3d_b200.box import box2d_nms, box2d_nms_batch
    rng = np.random.default_rng(17)
    sizes = (700, 0, 1, 64, 4096, 65, 1500, 333)
    frames = [proposals(rng, n, max(n // 20, 1), extent=30.0) if n else (np.zeros((0, 5)), np.zeros(0)) for n in sizes]
    for im, thr, sthr in (("rbox", 0.5, 0.0), ("rbox", 0.3, 0.2), ("box", 0.5, 0.1)):
        keeps = box2d_nms_batch([_t(b, dev) for b, _ in frames], [_t(s, dev) for _, s in frames], iou_method=im, iou_threshold=thr, score_threshold=sthr)
        assert len(keeps) == len(frames)
        for (b, s), k in zip(frames, keeps):
            assert k.dtype == torch.bool and k.shape == (len(b),)
            if len(b):
                single = box2d_nms(_t(b, dev), _t(s, dev), im, iou_threshold=thr, score_threshold=sthr)
                assert torch.equal(k, single), (im, len(b))
                if len(b) <= 1500:
                    assert np.array_equal(k.cpu().numpy(), oracle.box2d_nms(b, s, im, iou_threshold=thr, score_threshold=sthr, cuda_score_rule=True)), (im, len(b))
    packed_b = np.concatenate([b for b, _ in frames]).astype(np.float32)
    packed_s = np.concatenate([s for _, s in frames]).astype(np.float32)
    offs = np.concatenate([[0], np.cumsum(sizes)])
    k32 = box2d_nms_batch(packed_b, packed_s, offs, iou_method="rbox", iou_threshold=0.5, precise=False)     # numpy, packed, fp32
    assert isinstance(k32, np.ndarray) and k32.shape == (sum(sizes),)
    lo = 0
    for (b, s), n in zip(frames, sizes):
        if n:
            assert np.array_equal(k32[lo:lo + n], box2d_nms(b.astype(np.float32), s.astype(np.float32), "rbox", iou_threshold=0.5, precise=False)), n
        lo += n
    big = [proposals(rng, 9000, 300, extent=60.0), proposals(rng, 100, 5, extent=10.0)]                          # a frame beyond 8192 boxes: per-frame fallback
    kb = box2d_nms_batch([_t(b, dev) for b, _ in big], [_t(s, dev) for _, s in big], iou_method="rbox", iou_threshold=0.5)
    assert torch.equal(kb[0], box2d_nms(_t(big[0][0], dev), _t(big[0][1], dev), "rbox", iou_threshold=0.5))
    assert box2d_nms_batch([], []) == []
    # the two batched back ends for rotated boxes (Morton order + edge list + fixpoint | score order + dense matrix + walk) agree; a frame of
    # near-identical boxes overflows its edge list (n^2 / 2 edges) and the dense kernels behind the device flag redo the batch; equal scores
    # (ties go to the lower index) and a negative threshold (always the dense path: disjoint boxes suppress too)
    crowd = (np.tile(np.array([[1.0, 2.0, 3.0, 2.0, 0.3]]), (2500, 1)) + rng.normal(0, 1e-3, (2500, 5)), rng.random(2500))
    ties = (frames[0][0], np.round(frames[0][1] * 4) / 4)
    mixed = [frames[4], crowd, frames[6], ties]
    for thr in (0.5, -1.0):
        out = {}
        for path in (None, 1):
            _cabi.tuning_set("D3D_B200_NMS_BATCH_PATH", path)
            out[path] = box2d_nms_batch([_t(b, dev) for b, _ in mixed], [_t(s, dev) for _, s in mixed], iou_method="rbox", iou_threshold=thr)
        _cabi.tuning_set("D3D_B200_NMS_BATCH_PATH", None)
        for (b, s), k0, k1 in zip(mixed, out[None], out[1]):
            assert torch.equal(k0, k1), (thr, len(b))
            assert torch.equal(k0, box2d_nms(_t(b, dev), _t(s, dev), "rbox", iou_threshold=thr)), (thr, len(b))
    # the per-frame resolve of the edge path has two forms (pulled over predecessor lists in shared memory | rounds over the edge list,
    # the fallback of frames with too many edges): same masks; a 300-deep chain of alternating decisions in one frame
    m = 600
    chain = (np.stack([0.2 * np.arange(m), np.zeros(m), np.ones(m), np.ones(m), 0.37 * np.arange(m)], 1), rng.random(m))
    deep = [frames[4], chain, frames[6], frames[0]]
    got = {}
    for fix in (None, 2):
        _cabi.tuning_set("D3D_B200_NMS_FIX", fix)
        got[fix] = box2d_nms_batch([_t(b, dev) for b, _ in deep], [_t(s, dev) for _, s in deep], iou_method="rbox", iou_threshold=0.5)
    _cabi.tuning_set("D3D_B200_NMS_FIX", None)
    for (b, s), k0, k2 in zip(deep, got[None], got[2]):
        assert torch.equal(k0, k2), len(b)
        assert torch.equal(k0, box2d_nms(_t(b, dev), _t(s, dev), "rbox", iou_threshold=0.5)), len(b)
    assert np.array_equal(got[None][1].cpu().numpy(), oracle.box2d_nms(chain[0], chain[1], "rbox", iou_threshold=0.5, cuda_score_rule=True))


def test_nms_parallel_resolve_equals_list_walk(dev, oracle):
    """the resolve phase has two forms -- the block-by-block walk in score order on one SM and the parallel fixpoint pulled over transposed
    hit lists (default from 8192 boxes on) -- with the same keep mask: sizes on both sides of the switch, both candidate back ends, score
    thresholds, and a chain of pairwise overlapping boxes 200 decisions deep that both forms follow to the end"""
    from d3d_b200.box import box2d_nms
    rng = np.random.default_rng(11)
    cases = [proposals(rng, n, nobj, extent=ext) for n, nobj, ext in ((64, 4, 10.0), (1000, 30, 30.0), (4097, 150, 60.0), (12000, 500, 75.0))]
    m = 400   # unit squares 0.2 apart, each turned by 0.37 rad against the last: neighbours overlap with IoU 0.61, second neighbours with 0.39
    chain = np.stack([0.2 * np.arange(m), np.zeros(m), np.ones(m), np.ones(m), 0.37 * np.arange(m)], 1)   # -> keep, suppress, keep, ... 200 decisions deep
    cases.append((chain, np.linspace(1.0, 0.1, m)))
    cases.append((np.concatenate([chain, cases[1][0]]), np.concatenate([np.linspace(1.0, 0.1, m), cases[1][1]])))
    for P, sc in cases:
        for thr, sthr in ((0.5, 0.0), (0.3, 0.4)):
            exp = oracle.box2d_nms(P, sc, "rbox", iou_threshold=thr, score_threshold=sthr, cuda_score_rule=True)
            for path in (None, 1):          # spatial candidates | dense tiles
                for fix in (0, 1):          # list walk | parallel fixpoint, pulled
                    _cabi.tuning_set("D3D_B200_NMS_PATH", path)
                    _cabi.tuning_set("D3D_B200_NMS_FIX", fix)
                    got = box2d_nms(_t(P, dev), _t(sc, dev), "rbox", iou_threshold=thr, score_threshold=sthr).cpu().numpy()
                    assert np.array_equal(got, exp), (len(P), thr, sthr, path, fix, int((got != exp).sum()))
    _cabi.tuning_set("D3D_B200_NMS_PATH", None)
    _cabi.tuning_set("D3D_B200_NMS_FIX", None)


def test_sort_forms_agree(dev):
    """the stable radix sort has two forms -- five launches per pass (any size) and, up to 131 072 keys, every pass inside one
    cooperative launch (the NMS score sort) -- with the same order: NMS keep masks with tied scores (ties go to the lower index: the
    sort must be stable) and the sort back end of the voxelizer, at sizes around the tile (2048) and the switch"""
    from d3d_b200.box import box2d_nms
    from d3d_b200.voxel import VoxelGenerator
    rng = np.random.default_rng(21)
    for n in (1, 33, 2048, 2049, 20000, 131072, 131073):
        P, sc = proposals(rng, n, max(1, n // 25), extent=75.0)
        sc = np.round(sc * 64) / 64          # many equal scores
        out = []
        for coop in (0, 1, 2):               # 2: all eight passes in the cooperative launch; 1 (default): the high key half + run fix-up for double scores
            _cabi.tuning_set("D3D_B200_SORT_COOP", coop)
            out.append(box2d_nms(_t(P, dev), _t(sc, dev), "rbox", iou_threshold=0.5).cpu().numpy())
        _cabi.tuning_set("D3D_B200_SORT_COOP", None)
        assert np.array_equal(out[0], out[1]) and np.array_equal(out[0], out[2]), n
    # double scores that differ in the LOW half of their bits only: every box twice (the twins overlap fully, exactly one is kept: the one
    # with the larger score), twins a few ulps apart in a random direction -- the keep mask spells out the order of every pair
    from oracle import oracle as _o
    for n in (4000, 50000):
        Pb, sb = proposals(rng, n // 2, n // 2, extent=500.0)
        P = np.repeat(Pb, 2, axis=0)
        ulps = rng.integers(1, 2000, n // 2) * np.where(rng.random(n // 2) < 0.5, 1, -1)
        tw = (sb.view(np.int64) + ulps).view(np.float64)
        sc = np.stack([sb, tw], 1).reshape(-1)
        out = []
        for coop in (0, 1, 2):
            _cabi.tuning_set("D3D_B200_SORT_COOP", coop)
            out.append(box2d_nms(_t(P, dev), _t(sc, dev), "rbox", iou_threshold=0.5).cpu().numpy())
        _cabi.tuning_set("D3D_B200_SORT_COOP", None)
        assert np.array_equal(out[0], out[1]) and np.array_equal(out[0], out[2]), n
        twins = out[1].reshape(-1, 2)
        lone = twins.sum(1) == 1            # pairs no third box interferes with
        assert lone.mean() > 0.5 and np.array_equal(twins[lone, 0], (sb > tw)[lone]), n
        if n <= 4000:
            assert np.array_equal(out[1], _o.box2d_nms(P, sc, "rbox", iou_threshold=0.5, cuda_score_rule=True)), n
    pts = lidar(rng, 60000)
    res = []
    for coop in (0, 1):
        _cabi.tuning_set("D3D_B200_SORT_COOP", coop)
        gen = VoxelGenerator([0, 70.4, -40, 40, -3, 1], [1408, 1600, 40], max_points=5, max_points_filter="trim")
        gen.algo = "sort"
        res.append({k: v.cpu().numpy() for k, v in gen(_t(pts, dev)).items()})
    _cabi.tuning_set("D3D_B200_SORT_COOP", None)
    for k in res[0]:
        assert np.array_equal(res[0][k], res[1][k]), k


def test_nms_back_ends_agree(dev):
    """the NMS back ends (spatial candidate grid with a CTA per cell, dense tiles + list resolve, dense matrix + dense resolve) give the
    same keep mask (the knob is set through d3d_tuning_set: the environment is read once)"""
    from d3d_b200.box import box2d_nms
    rng = np.random.default_rng(5)
    for n, nobj, extent in ((20000, 800, 75.0), (3000, 40, 30.0), (700, 700, 400.0)):
        P, s = proposals(rng, n, nobj, extent=extent)
        for dt in (np.float64, np.float32):
            out = {}
            for path in ("", "tiles", "dense"):   # "": spatial grid, a CTA per cell (default)
                _cabi.tuning_set("D3D_B200_NMS_PATH", {"": None, "dense": 2, "tiles": 1}[path])
                out[path] = box2d_nms(_t(P.astype(dt), dev), _t(s.astype(dt), dev), "rbox", iou_threshold=0.45, precise=dt == np.float64).cpu().numpy()
            _cabi.tuning_set("D3D_B200_NMS_PATH", None)
            assert np.array_equal(out[""], out["dense"]) and np.array_equal(out["tiles"], out["dense"]), (n, dt)
            assert 0 < out[""].sum() < n
    # a negative threshold suppresses disjoint pairs too (IoU 0 > thr), like the reference: only the best box survives
    P, s = proposals(rng, 500, 50, extent=100.0)
    for path in (None, 2):
        _cabi.tuning_set("D3D_B200_NMS_PATH", path)
        k = box2d_nms(_t(P, dev), _t(s, dev), "rbox", iou_threshold=-0.5).cpu().numpy()
        assert k.sum() == 1 and k[np.argmax(s)]
    _cabi.tuning_set("D3D_B200_NMS_PATH", None)


def test_nms_c3_scale_properties(dev, oracle):
    """config C3: 50k clustered proposals, rbox thr 0.5, fp64: the full keep mask against the fixture written by the reference's own
    CPU nms2d (one ~25 s run, committed as 6 KB of bits), NMS invariants, and a live oracle run on a prefix in score order."""
    from d3d_b200.box import box2d_nms, box2d_iou
    rng = np.random.default_rng(2)
    P, s = proposals(rng, 50000, 2000)
    tP, ts = _t(P, dev), _t(s, dev)
    keep = box2d_nms(tP, ts, "rbox", iou_threshold=0.5)
    k = keep.cpu().numpy()
    assert 3000 < k.sum() < 8000
    # invariant 1: kept boxes do not suppress each other
    kb = tP[keep]
    iou = box2d_iou(kb, kb, "rbox")
    iou.fill_diagonal_(0)
    assert float(iou.max()) <= 0.5
    # invariant 2: every suppressed box overlaps (> thr) a kept box with a higher score
    sb, ss = tP[~keep], ts[~keep]
    cross = box2d_iou(sb, kb, "rbox")
    higher = ts[keep][None, :] > ss[:, None]
    assert bool(((cross > 0.5) & higher).any(dim=1).all())
    # idempotence: NMS of the kept set keeps everything
    assert bool(box2d_nms(kb, ts[keep], "rbox", iou_threshold=0.5).all())
    # oracle on the 6000 best-scoring proposals (greedy NMS on a score prefix equals the prefix of the full run)
    top = np.argsort(-s, kind="stable")[:6000]
    assert np.array_equal(k[top], oracle.box2d_nms(P[top], s[top], "rbox", iou_threshold=0.5))
    # the full 50k mask, bit for bit, against the one written by the reference's own CPU nms2d (tests/golden/make_golden.py write_nms_c3)
    assert np.array_equal(k, _unpack(golden("nms_c3.npz")["keep"], 50000))


# ------------------------------------------------------------------ voxelization
VOX_CASES = {
    "sp_default": dict(), "sp_trim5": dict(max_points=5, max_points_filter="trim"),
    "sp_trim2_v1000": dict(max_points=2, max_points_filter="trim", max_voxels=1000, max_voxels_filter="trim"),
    "sp_min2": dict(min_points=2, max_points=3, max_points_filter="trim"),
    "de_p5": dict(dense=True, max_points=5, max_voxels=20000), "de_p2_v1000": dict(dense=True, max_points=2, max_voxels=1000),
    "de_mean": dict(dense=True, max_points=3, max_voxels=20000, reduction="mean"),
    "de_max": dict(dense=True, max_points=3, max_voxels=20000, reduction="max"),
    "de_min": dict(dense=True, max_points=3, max_voxels=700, reduction="min"),
}
EXPECT_DTYPES = dict(points=torch.float32, points_mask=torch.int64, points_mapping=torch.int64, voxel_npoints=torch.int32,
                     coords=torch.int64, voxels=torch.float32, voxel_pmask=torch.bool, aggregates=torch.float32)


@pytest.fixture(autouse=True, params=["auto", "sort", "auto_no_tiles"])
def voxel_backend(request):
    """every voxel test runs on all back ends: "auto" (tile pipeline wherever it supports the configuration, else as
    below), "auto_no_tiles" (cluster-per-frame hash path wherever it supports the configuration) and "sort" (the
    general pipeline); the outputs must be bit-identical"""
    if "voxel" not in request.node.name:
        if request.param != "auto":
            pytest.skip("back-end parameter only applies to the voxel tests")
        yield
        return
    from d3d_b200.voxel import VoxelGenerator
    VoxelGenerator.default_algo = request.param
    yield
    VoxelGenerator.default_algo = "auto"


def _cmp_vox(r, exp, kw, tag):
    assert set(r.keys()) == set(exp.keys()), (tag, r.keys(), exp.keys())
    for k, v in exp.items():
        got = r[k]
        assert got.dtype == EXPECT_DTYPES[k], (tag, k, got.dtype)
        got = got.cpu().numpy()
        if k == "voxel_pmask":
            P = kw["max_points"]
            sl = np.arange(P)[None, :] < np.minimum(exp["voxel_npoints"], P)[:, None]
            assert got.shape == v.shape and np.array_equal(got[sl], v[sl]) and not got[~sl].any(), (tag, k)
        else:
            assert got.shape == v.shape and np.array_equal(got, v), (tag, k)


def test_voxel_spconv_golden(dev):
    """test/test_voxel.py:80-88 with test/voxel_data.npz (spconv VoxelGeneratorV2)."""
    from d3d_b200.voxel import VoxelGenerator
    d = golden("voxel_spconv.npz")
    gen = VoxelGenerator([0, 1, 0, 1, 0, 1], [10, 10, 10], max_points=5, max_points_filter="trim", dense=True)
    for cloud in (_t(d["cloud"], dev), torch.from_numpy(d["cloud"])):   # CUDA and host input
        ret = gen(cloud)
        assert np.array_equal(ret.voxels.cpu().numpy(), d["voxels"])
        assert np.array_equal(ret.coords.cpu().numpy(), d["coords"])


def test_voxel_golden_fixtures(dev):
    from d3d_b200.voxel import VoxelGenerator
    g = golden("voxel_c2small.npz")
    pts = g["points"]
    for name, kw in VOX_CASES.items():
        r = VoxelGenerator(g["bounds"].tolist(), g["shape"].tolist(), **kw)(_t(pts, dev))
        exp = {}
        for key in g.files:
            if key.startswith(name + "."):
                k = key.split(".", 1)[1]
                v = g[key]
                if k == "voxel_pmask":
                    shp = (len(g[f"{name}.voxel_npoints"]), kw["max_points"])
                    v = np.unpackbits(v)[:shp[0] * shp[1]].reshape(shp).astype(bool)
                exp[k] = v
        if not kw.get("dense"):
            exp["points"] = pts[exp["points_mask"]]
        _cmp_vox(r, exp, kw, name)
    for name, kw in {"co_trim5": dict(max_points=5, max_points_filter="trim"),
                     "co_de_mean": dict(dense=True, max_points=4, max_voxels=300, reduction="mean")}.items():
        r = VoxelGenerator(g["coarse_bounds"].tolist(), g["coarse_shape"].tolist(), **kw)(_t(pts, dev))
        exp = {}
        for key in g.files:
            if key.startswith(name + "."):
                k = key.split(".", 1)[1]
                v = g[key]
                if k == "voxel_pmask":
                    shp = (len(g[f"{name}.voxel_npoints"]), kw["max_points"])
                    v = np.unpackbits(v)[:shp[0] * shp[1]].reshape(shp).astype(bool)
                exp[k] = v
        if not kw.get("dense"):
            exp["points"] = pts[exp["points_mask"]]
        _cmp_vox(r, exp, kw, name)


def test_voxel_c2_full_vs_oracle(dev, oracle):
    """config C2 (120k points, KITTI grid) and C3 cloud (180k, 3008^2 x 60 grid), every mode, bit-exact."""
    from d3d_b200.voxel import VoxelGenerator
    pts = lidar(np.random.default_rng(1), 120000)
    bounds, shape = [0, 70.4, -40, 40, -3, 1], [1408, 1600, 40]
    cases = [dict(max_points=5, max_points_filter="trim"),
             dict(max_points=5, max_points_filter="trim", max_voxels=20000, max_voxels_filter="trim"), dict(),
             dict(min_points=2, max_points=3, max_points_filter="trim"),
             dict(dense=True, max_points=5, max_voxels=20000), dict(dense=True, max_points=5, max_voxels=200000),
             dict(dense=True, max_points=5, max_voxels=20000, reduction="mean"),
             dict(dense=True, max_points=3, max_voxels=20000, reduction="max")]
    for kw in cases:
        r = VoxelGenerator(bounds, shape, **kw)(_t(pts, dev))
        _cmp_vox(r, oracle.VoxelGenerator(bounds, shape, **kw)(pts), kw, str(kw))
    r = VoxelGenerator(bounds, shape, max_points=5, max_points_filter="trim")(_t(pts, dev))
    assert len(r.coords) == 81559 and len(r.points) == 85387        # SURVEY Appendix C anchors
    rng = np.random.default_rng(2)
    n = 180000
    rho = 75 * rng.random(n) ** 2; th = (rng.random(n) - .5) * 2 * np.pi
    p3 = np.stack([rho * np.cos(th), rho * np.sin(th), rng.normal(-1.2, .6, n), rng.random(n)], 1).astype(np.float32)
    b3, s3 = [-75.2, 75.2, -75.2, 75.2, -2, 4], [3008, 3008, 60]
    for kw in (dict(max_points=5, max_points_filter="trim"), dict(dense=True, max_points=5, max_voxels=40000)):
        _cmp_vox(VoxelGenerator(b3, s3, **kw)(_t(p3, dev)), oracle.VoxelGenerator(b3, s3, **kw)(p3), kw, "c3 " + str(kw))


def test_voxel_descending_and_crowded(dev, oracle):
    """coarse grid: many points per voxel (trim, ordered MEAN sums), DESCENDING with tie rule = ascending id"""
    from d3d_b200.voxel import VoxelGenerator
    pts = lidar(np.random.default_rng(8), 30000)
    b, s = [0, 70.4, -40, 40, -3, 1], [44, 50, 4]
    for kw in (dict(max_points=5, max_points_filter="trim"), dict(max_points=1, max_points_filter="trim"), dict(max_points=2, max_points_filter="trim"),
               dict(max_points=8, max_points_filter="trim"), dict(max_points=7, max_points_filter="trim", max_voxels=60, max_voxels_filter="trim"),
               dict(max_voxels=50, max_voxels_filter="descending", min_points=3),
               dict(max_voxels=5000, max_voxels_filter="descending", max_points=4, max_points_filter="trim"),
               dict(dense=True, max_points=4, max_voxels=300, reduction="mean"), dict(dense=True, max_points=9, max_voxels=9000, reduction="min")):
        _cmp_vox(VoxelGenerator(b, s, **kw)(_t(pts, dev)), oracle.VoxelGenerator(b, s, **kw)(pts), kw, "crowded " + str(kw))
    # every point in ONE voxel (worst case for per-voxel work) and an empty / all-outside cloud
    one = np.tile(np.array([[10.01, 0.01, -1.01, 0.5]], np.float32), (5000, 1)); one[:, 3] = np.arange(5000)
    for kw in (dict(max_points=5, max_points_filter="trim"), dict(dense=True, max_points=5, max_voxels=10, reduction="mean")):
        _cmp_vox(VoxelGenerator(b, s, **kw)(_t(one, dev)), oracle.VoxelGenerator(b, s, **kw)(one), kw, "one-voxel")
    out = np.full((100, 4), 500.0, np.float32)
    r = VoxelGenerator(b, s)(_t(out, dev))
    assert len(r.points) == 0 and len(r.coords) == 0 and r.coords.shape == (0, 3)
    r = VoxelGenerator(b, s)(torch.zeros((0, 4), device=dev))
    assert len(r.points) == 0 and len(r.voxel_npoints) == 0
    nan = lidar(np.random.default_rng(3), 1000); nan[::7, 1] = np.nan; nan[5::11, 0] = np.inf
    for kw in (dict(), dict(dense=True, max_points=3, max_voxels=500)):
        _cmp_vox(VoxelGenerator(b, s, **kw)(_t(nan, dev)), oracle.VoxelGenerator(b, s, **kw)(nan), kw, "nan")


def test_voxel_reference_tests(dev):
    """test/test_voxel.py:11-78 ported verbatim in spirit (dense + sparse semantic pins, filters)."""
    from d3d_b200.voxel import VoxelGenerator
    cloud = torch.rand((2000, 4), dtype=torch.float32)
    cloud = torch.cat((cloud, torch.tensor([[-1, -1, -1, -100], [-2, -2, -2, 100]], dtype=torch.float32)), axis=0)
    gen = VoxelGenerator([0, 1, 0, 1, 0, 1], [10, 10, 10], reduction="mean", max_points=5, max_voxels=20000,
                         max_points_filter="trim", max_voxels_filter="trim", dense=True)
    data = gen(cloud.to(dev))
    assert len(data.voxels) == len(data.coords) and len(data.voxels) <= 1000
    assert torch.all((data.voxels >= 0) & (data.voxels <= 1)) and torch.all((data.coords >= 0) & (data.coords <= 10))
    v, c, n = data.voxels.cpu(), data.coords.cpu(), data.voxel_npoints.cpu()
    for i in range(len(v)):
        for j in range(min(int(n[i]), 5)):
            for k in range(3):
                assert c[i, k] == int(v[i, j, k] * 10)
    gen = VoxelGenerator([0, 1, 0, 1, 0, 1], [10, 10, 10], reduction="none", max_points=5, max_voxels=20000,
                         max_points_filter="trim", max_voxels_filter="trim", dense=True)
    data = gen(cloud.to(dev))
    assert 'aggregates' not in data and len(data.voxels) == len(data.coords)
    data = VoxelGenerator([0, 1, 0, 1, 0, 1], [10, 10, 10])(cloud)       # host tensor in, host tensors out
    assert len(data.points) == 2000 and len(data.coords) <= 1000 and not data.points.is_cuda
    assert torch.equal(data.coords[data.points_mapping], (cloud[:2000, :3] * 10).long())
    cloud3 = (torch.rand((2000, 3), dtype=torch.float32) - 0.5) * 4
    data = VoxelGenerator([-1, 1, -1, 1, -1, 1], [20, 20, 20])(cloud3.to(dev))
    assert torch.all((data.points >= -1) & (data.points <= 1)) and torch.all((data.coords >= 0) & (data.coords <= 20))
    assert torch.equal(data.coords[data.points_mapping], ((data.points + 1) * 10).long())
    assert len(VoxelGenerator([0, 1, 0, 1, 0, 1], [10, 10, 10], max_voxels=10, max_voxels_filter="trim")(cloud3.to(dev)).coords) <= 10
    assert len(VoxelGenerator([0, 1, 0, 1, 0, 1], [10, 10, 10], max_voxels=10, max_voxels_filter="descending")(cloud3.to(dev)).coords) <= 10
    data = VoxelGenerator([0, 1, 0, 1, 0, 1], [10, 10, 10], min_points=2, max_points=4, max_points_filter="trim")(cloud3.to(dev))
    assert torch.all((data.voxel_npoints >= 2) & (data.voxel_npoints <= 4))
    with pytest.raises(ValueError):
        VoxelGenerator([0.013, 1, 0, 1, 0, 1], [10, 10, 10])
    with pytest.raises(ValueError):
        VoxelGenerator([0, 1, 0, 1, 0, 1], [10, 10, 10], reduction="mean")
    with pytest.raises(NotImplementedError):
        VoxelGenerator([0, 1, 0, 1, 0, 1], [10, 10, 10], max_points_filter="farthest_sampling")(cloud3.to(dev))
    gen = VoxelGenerator([0, 1, 0, 1, 0, 1], [10, 10, 10], max_voxels=10, max_voxels_filter="descending")
    gen.algo = "cluster"                      # the cluster back end does not order voxels by count: explicit request fails
    with pytest.raises(NotImplementedError):
        gen(cloud3.to(dev))


def test_voxel_batch_equals_per_frame(dev, oracle):
    """frame batching (C5): one launch sequence over 6 ragged frames == 6 independent calls == oracle"""
    from d3d_b200.voxel import VoxelGenerator
    frames = [lidar(np.random.default_rng(100 + i), n) for i, n in enumerate((9000, 1, 0, 12000, 777, 4096))]
    bounds, shape = [0, 70.4, -40, 40, -3, 1], [352, 400, 40]
    for kw in (dict(max_points=3, max_points_filter="trim", max_voxels=2500, max_voxels_filter="trim"),
               dict(max_voxels=300, max_voxels_filter="descending", min_points=2),
               dict(dense=True, max_points=4, max_voxels=3000, reduction="mean")):
        gen = VoxelGenerator(bounds, shape, **kw)
        res = gen.batch([_t(f, dev) for f in frames])
        for f, r in zip(frames, res):
            _cmp_vox(r, oracle.VoxelGenerator(bounds, shape, **kw)(f), kw, "batch " + str(kw))


def test_voxel_routed_and_l2_frames_in_one_launch(dev):
    """one batch whose frames take different per-frame back ends inside the same persistent launch: routed (fits the cluster's
    shared memory), L2 (more than 131072 points), routed-then-bailed (40 % of the points in one cell: queue overflow) --
    packed outputs and per-frame results equal the sort pipeline's"""
    from d3d_b200.voxel import VoxelGenerator
    rng = np.random.default_rng(77)
    sizes = (120000, 140000, 3000, 131072, 150000, 60000, 1, 90000)
    frames = [lidar(rng, n) for n in sizes]
    frames[5][rng.integers(0, 60000, 24000)] = np.array([10.01, 0.01, -1.0, 0.5], np.float32)
    bounds, shape = [0, 70.4, -40, 40, -3, 1], [1408, 1600, 40]
    for kw in (dict(max_points=5, max_points_filter="trim"), dict(max_points=3, max_points_filter="trim", max_voxels=30000, max_voxels_filter="trim", min_points=2)):
        out = {}
        for algo in ("cluster", "sort"):
            gen = VoxelGenerator(bounds, shape, **kw)
            gen.algo = algo
            out[algo] = gen.batch([_t(f, dev) for f in frames])
        for a, b in zip(out["cluster"], out["sort"]):
            assert set(a.keys()) == set(b.keys())
            for k in a:
                assert torch.equal(a[k], b[k]), (kw, k)


def test_box_pdist_vs_truth_and_reference(dev, oracle):
    """f4: signed point-to-rotated-box distance.  Forward against the local-frame truth (oracle.pdist2dr_local) on every pair, and
    against the fixture written by the reference's own pdist2dr_forward and the oracle's restatement of it where the reference agrees
    with the truth (deviation P1 of SURVEY.md 8(c): it does not on points on the lines through edges and at headings of pi / 2).
    Backward against five-point differences of the truth, and point gradients against the reference's on the points whose every pair
    the reference gets right; 3-D wrapper against the local combination of the same terms."""
    from d3d_b200.box import box2dr_pdist, box3dr_pdist
    g = golden("pdist.npz")
    for tag, tol in (("f32", 1e-5), ("f64", 1e-10)):
        pts, bx = g[f"{tag}.points"], g[f"{tag}.boxes"]
        d = box2dr_pdist(_t(pts, dev), _t(bx, dev))
        assert d.shape == (len(bx), len(pts)) and d.dtype == _t(pts, dev).dtype
        d, truth = d.cpu().numpy(), oracle.pdist2dr_local(pts, bx)
        sane = np.abs(g[f"{tag}.dist"] - truth) <= tol
        assert sane.mean() > 0.99 and np.array_equal(oracle.pdist2dr(pts, bx), g[f"{tag}.dist"]), tag
        assert np.abs(d - truth).max() < tol and np.abs(d - g[f"{tag}.dist"])[sane].max() < 2 * tol, tag
    pnp, bnp, up = g["f64.points"], g["f64.boxes"], g["f64.grad"]
    v, dp, db, smooth = oracle.pdist2dr_grad_local(pnp, bnp)
    sane = np.abs(g["f64.dist"] - v) <= 1e-9
    # the reference's point gradients where all 24 pairs of a point are right and differentiable
    cols = (sane & smooth).all(0)
    pts, bx = _t(pnp, dev).requires_grad_(True), _t(bnp, dev).requires_grad_(True)
    (box2dr_pdist(pts, bx) * _t(up, dev)).sum().backward()
    assert cols.mean() > 0.9 and np.abs(pts.grad.cpu().numpy() - g["f64.grad_points"])[cols].max() < 1e-9
    upm = up * smooth
    pts, bx = _t(pnp, dev).requires_grad_(True), _t(bnp, dev).requires_grad_(True)
    (box2dr_pdist(pts, bx) * _t(upm, dev)).sum().backward()
    assert smooth.mean() > 0.99
    assert np.abs(pts.grad.cpu().numpy() - np.einsum("ij,ijk->jk", upm, dp)).max() < 1e-8
    assert np.abs(bx.grad.cpu().numpy() - np.einsum("ij,ijk->ik", upm, db)).max() < 1e-8
    rng = np.random.default_rng(13)
    for n, m in ((1, 1), (1000, 9), (257, 70)):
        p, b = (rng.random((n, 2)) - .5) * 14, gen_boxes(rng, m)
        od = box2dr_pdist(torch.from_numpy(p), torch.from_numpy(b)).numpy()   # host tensors in, host tensor out
        assert np.abs(od - oracle.pdist2dr_local(p, b)).max() < 1e-10
    p3 = (rng.random((400, 3)) - .5) * 10
    b3 = np.concatenate([gen_boxes(rng, 15)[:, :2], rng.random((15, 1)), rng.random((15, 3)) * 4 + .2, rng.random((15, 1)) * 6], 1)
    for ax in (0, 1, 2):
        d3 = box3dr_pdist(_t(p3, dev), _t(b3, dev), ax).cpu().numpy()
        truth = oracle.box3dr_pdist_local(p3, b3, ax)
        sane = np.abs(oracle.box3dr_pdist(p3, b3, ax) - truth) <= 1e-9
        assert sane.mean() > 0.99 and np.abs(d3 - truth).max() < 1e-10 and np.abs(d3 - oracle.box3dr_pdist(p3, b3, ax))[sane].max() < 1e-10
    with pytest.raises(ValueError):
        box2dr_pdist(_t(pnp, dev), _t(bnp, dev), method="box")
    assert box2dr_pdist(torch.zeros((0, 2), dtype=torch.float64, device=dev), _t(bnp, dev)).shape == (len(bnp), 0)


# ------------------------------------------------------------------ aligned scatter
def test_scatter_golden_and_oracle(dev, oracle):
    from d3d_b200.point import aligned_scatter
    g = golden("scatter.npz")
    for tag in ("f32", "f64"):
        for dim in (1, 2, 3):
            img, crd = g[f"{tag}.d{dim}.image"], g[f"{tag}.d{dim}.coord"]
            for meth, at in (("mean", 1), ("linear", 2)):
                out = aligned_scatter(_t(crd, dev), _t(img, dev), meth).cpu().numpy()
                assert out.dtype == img.dtype and np.array_equal(out, g[f"{tag}.d{dim}.{meth}"]), (tag, dim, meth)
                # backward against the oracle (reference CPU backward is a no-op at this commit, see make_golden.py)
                ti = _t(img, dev).requires_grad_(True)
                o = aligned_scatter(_t(crd, dev), ti, meth)
                gr = np.random.default_rng(dim).random(o.shape).astype(img.dtype)
                o.backward(_t(gr, dev))
                exp = oracle.scatter_backward(crd, gr, at, img.shape)
                tol = 1e-5 if tag == "f32" else 1e-12   # atomics add in arbitrary order
                assert np.abs(ti.grad.cpu().numpy() - exp).max() < tol, (tag, dim, meth)


def test_scatter_reference_test(dev):
    """test/test_point.py:10-69 (drop / mean / linear forward and backward known answers)"""
    from d3d_b200.point import aligned_scatter
    coord = torch.tensor([[0, 0.25, 0.25, 0.25], [0, 1.25, 1.25, 1.25], [1, 2.25, 2.25, 2.25]], device=dev)
    image_feat = torch.rand(2, 10, 3, 3, 3, device=dev)
    image_feat.requires_grad = True
    indexing = lambda icoord: (icoord[:, 0], slice(None)) + tuple(icoord[:, i] for i in range(1, coord.shape[1]))
    lcoords = torch.tensor(np.array(np.meshgrid([0, 1], [0, 1], [0, 1])).T.reshape(-1, 3), device=dev)
    pfeat = aligned_scatter(coord, image_feat, "drop")
    assert torch.allclose(pfeat, image_feat[indexing(coord.long())])
    pfeat.sum().backward()
    assert torch.allclose(image_feat.grad[0, :, 0, 0, 0], torch.full([10], 1.0, device=dev))
    pfeat = aligned_scatter(coord, image_feat, "mean")
    icoord = torch.cat([torch.full((8, 1), 0, dtype=torch.long, device=dev), lcoords], dim=1)
    assert torch.allclose(pfeat[0], torch.mean(image_feat[indexing(icoord)], dim=0))
    icoord = torch.cat([torch.full((8, 1), 0, dtype=torch.long, device=dev), lcoords + 1], dim=1)
    assert torch.allclose(pfeat[1], torch.mean(image_feat[indexing(icoord)], dim=0))
    assert torch.allclose(pfeat[2], image_feat[1, :, 2, 2, 2])
    image_feat.grad.zero_()
    pfeat.sum().backward()
    assert torch.allclose(image_feat.grad[0, :, 0, 0, 0], torch.full([10], 1 / 8, device=dev))
    assert torch.allclose(image_feat.grad[0, :, 1, 1, 1], torch.full([10], 1 / 4, device=dev))
    assert torch.allclose(image_feat.grad[1, :, 2, 2, 2], torch.full([10], 1.0, device=dev))
    pfeat = aligned_scatter(coord, image_feat, "linear")
    nhigh = torch.sum(lcoords, dim=1).long()
    wmap = torch.tensor([0.25 ** i * 0.75 ** (3 - i) for i in range(4)], device=dev)
    lweight = wmap[nhigh]
    icoord = torch.cat([torch.full((8, 1), 0, dtype=torch.long, device=dev), lcoords], dim=1)
    assert torch.allclose(pfeat[0], torch.sum(image_feat[indexing(icoord)] * lweight.unsqueeze(1), dim=0))
    assert torch.allclose(pfeat[2], image_feat[1, :, 2, 2, 2])
    image_feat.grad.zero_()
    pfeat.sum().backward()
    assert torch.allclose(image_feat.grad[0, :, 0, 0, 0], torch.full([10], .75 ** 3, device=dev))
    assert torch.allclose(image_feat.grad[0, :, 1, 1, 1], torch.full([10], .75 ** 3 + .25 ** 3, device=dev))
    assert torch.allclose(image_feat.grad[1, :, 2, 2, 2], torch.full([10], 1.0, device=dev))
    with pytest.raises(AttributeError):
        aligned_scatter(coord, image_feat, "bogus")
    with pytest.raises(ValueError):
        aligned_scatter(coord, image_feat, "max")


def test_scatter_c2s_anchor(dev, oracle):
    """SURVEY 8(d) C2s: 88k points x 64 channels from a 1x64x704x800 map; checksum anchors + sampled oracle rows"""
    from d3d_b200.point import aligned_scatter
    pts = lidar(np.random.default_rng(1), 120000)
    sel = (pts[:, 0] >= 0) & (pts[:, 0] < 70.4) & (pts[:, 1] >= -40) & (pts[:, 1] < 40)
    p = pts[sel]
    crd = np.stack([np.zeros(len(p), np.float32), p[:, 0] / np.float32(0.1), (p[:, 1] + np.float32(40)) / np.float32(0.1)], 1).astype(np.float32)
    fm = torch.rand((1, 64, 704, 800), generator=torch.Generator().manual_seed(7))
    tf, tc = fm.to(dev), _t(crd, dev)
    om, ol = aligned_scatter(tc, tf, "mean"), aligned_scatter(tc, tf, "linear")
    if len(p) == 88596:
        assert abs(om.double().sum().item() - 2835634.619722) < 0.5 and abs(ol.double().sum().item() - 2834503.070217) < 0.5
    idx = np.random.default_rng(0).integers(0, len(p), 200)
    fmn = fm.numpy()
    assert np.array_equal(om.cpu().numpy()[idx], oracle.scatter_forward(crd[idx], fmn, 1))
    assert np.array_equal(ol.cpu().numpy()[idx], oracle.scatter_forward(crd[idx], fmn, 2))
    # full size, both back ends: the default above is the tile path (TMA); the gather path must give the same bits, and the two
    # backward passes the same map gradient up to the order of their sums
    grads = {}
    for path in (1, 2):
        _cabi.tuning_set("D3D_B200_SCATTER_PATH", path)
        tfg = tf.clone().requires_grad_(True)
        o = aligned_scatter(tc, tfg, "linear")
        assert torch.equal(o.detach(), ol), path
        o.backward(torch.ones_like(o))
        grads[path] = tfg.grad
    _cabi.tuning_set("D3D_B200_SCATTER_PATH", None)
    assert float((grads[1] - grads[2]).abs().max()) < 1e-3 * max(1.0, float(grads[1].abs().max()))
    assert abs(float(grads[2].double().sum()) - 64.0 * len(p)) < 1e-3 * 64.0 * len(p)   # every point spreads weight 1 per channel (up to the 2x quirk on integral coordinates: none here)


def test_scatter_tile_path_equals_gather_and_oracle(dev, oracle):
    """the tile path (2-D fp32 maps staged tile by tile in shared memory) against the gather path and the oracle: forward bit for bit, backward
    to rounding; ragged map sizes (tiles cut by the border, widths that are no multiple of 4), several batch images, channel counts that
    are no multiple of the 32-channel chunk, coordinates outside the map and on integers, a tile holding thousands of points (slices)"""
    from d3d_b200.point import aligned_scatter
    rng = np.random.default_rng(5)
    for (nb, ch, H, W, n) in ((1, 64, 64, 128, 6000), (2, 40, 37, 131, 5000), (1, 3, 9, 65, 900), (3, 33, 8, 64, 2000), (1, 32, 70, 200, 20000)):
        img = rng.random((nb, ch, H, W), dtype=np.float32)
        crd = np.stack([rng.integers(0, nb, n).astype(np.float32), rng.random(n, dtype=np.float32) * (H + 2) - 1, rng.random(n, dtype=np.float32) * (W + 2) - 1], 1)
        crd[: n // 10, 1:] = np.round(crd[: n // 10, 1:])                      # integral coordinates: the 2x weight quirk
        crd[n // 10: n // 5, 1:] = crd[n // 10: n // 5, 1:] * 0.05 + 3.0        # a crowd inside one tile
        for meth, at in (("mean", 1), ("linear", 2)):
            res = {}
            for path in (1, 2):
                _cabi.tuning_set("D3D_B200_SCATTER_PATH", path)
                ti = _t(img, dev).requires_grad_(True)
                o = aligned_scatter(_t(crd, dev), ti, meth)
                gr = np.random.default_rng(n).random(o.shape).astype(np.float32)
                o.backward(_t(gr, dev))
                res[path] = (o.detach().cpu().numpy(), ti.grad.cpu().numpy())
            _cabi.tuning_set("D3D_B200_SCATTER_PATH", None)
            assert np.array_equal(res[1][0], res[2][0]), (nb, ch, H, W, meth)
            sel = rng.integers(0, n, 300)
            assert np.array_equal(res[2][0][sel], oracle.scatter_forward(crd[sel], img, at)), (nb, ch, H, W, meth)
            exp = oracle.scatter_backward(crd, gr, at, img.shape)
            scale = max(1.0, float(np.abs(exp).max()))
            assert np.abs(res[2][1] - exp).max() < 2e-5 * scale and np.abs(res[1][1] - exp).max() < 2e-5 * scale, (nb, ch, H, W, meth)
    # the default rule picks the tile path for a dense cloud and the gather path for a sparse one; both give the oracle's rows
    img = rng.random((1, 8, 64, 64), dtype=np.float32)
    for n in (10, 4000):
        crd = np.stack([np.zeros(n, np.float32), rng.random(n, dtype=np.float32) * 63, rng.random(n, dtype=np.float32) * 63], 1)
        assert np.array_equal(aligned_scatter(_t(crd, dev), _t(img, dev), "linear").cpu().numpy(), oracle.scatter_forward(crd, img, 2))


@pytest.mark.gpu
def test_voxel_rank_paths_stress(dev, oracle):
    """the three rank regimes of the cluster back end (voxels with <= max_points points, up to 32, beyond 32) in
    one frame, zero-padded clouds (thousands of identical points), max_points 0 / 1 / large, ragged batches"""
    from d3d_b200.voxel import VoxelGenerator
    rng = np.random.default_rng(21)
    pts = lidar(rng, 40000)
    pts[rng.integers(0, len(pts), 6000)] = np.array([0.5, 0.5, -0.5, 0], np.float32)   # padding-like duplicates
    pts[:, 3] = np.arange(len(pts)) % 977                                                # feature identifies the point
    b, s = [0, 70.4, -40, 40, -3, 1], [176, 200, 8]
    cases = [dict(max_points=k, max_points_filter="trim") for k in (0, 1, 5, 33, 200)]
    cases += [dict(max_points=5, max_points_filter="trim", min_points=3, max_voxels=700, max_voxels_filter="trim"),
              dict(dense=True, max_points=0, max_voxels=100), dict(dense=True, max_points=1, max_voxels=30000),
              dict(dense=True, max_points=40, max_voxels=2000), dict(dense=True, max_points=7, max_voxels=35000)]
    for kw in cases:
        _cmp_vox(VoxelGenerator(b, s, **kw)(_t(pts, dev)), oracle.VoxelGenerator(b, s, **kw)(pts), kw, "stress " + str(kw))
    frames = [pts[:n] for n in (40000, 33, 0, 1025, 8192, 1, 20000, 31, 17000, 64, 5, 12345, 2, 30000, 999, 4097, 7, 26000, 513, 3000)]
    for kw in (dict(max_points=5, max_points_filter="trim"), dict(dense=True, max_points=3, max_voxels=5000)):
        gen = VoxelGenerator(b, s, **kw)
        for f, r in zip(frames, gen.batch([_t(f, dev) for f in frames])):
            _cmp_vox(r, oracle.VoxelGenerator(b, s, **kw)(f), kw, "ragged batch " + str(kw))
    p3 = pts[:, :3].copy()                                                                # nfeat = 3 (no float4 path)
    _cmp_vox(VoxelGenerator(b, s, max_points=2, max_points_filter="trim")(_t(p3, dev)),
             oracle.VoxelGenerator(b, s, max_points=2, max_points_filter="trim")(p3), dict(max_points=2), "nfeat3")
