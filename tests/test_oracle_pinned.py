"""Pin the CPU oracle (oracle/d3d_oracle.c) against the reference: its own golden vectors and
known-answer tests, fixtures generated from its compiled CPU extensions (tests/golden/make_golden.py),
and -- when oracle/_ref is present -- the reference extensions live.  CPU only."""
import numpy as np

from conftest import golden, gen_boxes, SOFT_CASES, SOFT_TEST6, soft_inputs
from conftest import LIVE_VOXEL, assert_pinned, live_dist3d_inputs, live_iou_nms_voxel_inputs, live_pdist_inputs


def _unpack(bits, n):
    return np.unpackbits(bits)[:n].astype(bool)


# ------------------------------------------------------------------ IoU
def test_iou_rc_bit_exact_vs_reference_fixture(oracle):
    g = golden("iou_c1.npz")
    a, b = g["boxes1"], g["boxes2"]
    assert np.array_equal(oracle.iou2dr(a, b, oracle.ALG_RC), g["rbox_f64"])
    assert np.array_equal(oracle.iou2d(a, b), g["box_f64"])
    a32, b32 = a.astype(np.float32), b.astype(np.float32)
    # fp32 goes through libm sinf/cosf/atan2f: identical on the same glibc, else within tolerance
    assert np.allclose(oracle.iou2dr(a32, b32, oracle.ALG_RC), g["rbox_f32"], atol=1e-4)
    assert np.allclose(oracle.iou2d(a32, b32), g["box_f32"], atol=1e-5)


def test_iou_c1_anchors(oracle):
    """SURVEY Appendix C anchors for config C1 (1k x 1k fp64)."""
    rng = np.random.default_rng(0)
    A, B = gen_boxes(rng, 1000), gen_boxes(rng, 1000)
    r = oracle.iou2dr(A, B, oracle.ALG_RC)
    g = golden("iou_c1.npz")
    assert abs(r.sum() - float(g["c1_rbox_sum"])) < 1e-7
    assert (r != 0).sum() == int(g["c1_rbox_nnz"]) == 205623
    assert abs(oracle.iou2d(A, B).sum() - float(g["c1_box_sum"])) < 1e-7
    # the three algorithms agree in generic position (SURVEY F4: <= 1.3e-13)
    assert np.abs(oracle.iou2dr(A, B, oracle.ALG_SH) - r).max() < 1e-10
    assert np.abs(oracle.iou2dr_truth(A, B) - r).max() < 1e-10


def test_iou_reference_known_answers(oracle):
    """test/test_box.py:12-100 with the reference's own tolerances."""
    g = golden("iou_known_answers.npz")
    eps = 1e-3
    for alg in (oracle.ALG_RC, oracle.ALG_TRUTH):
        assert np.allclose(oracle.box2d_iou(g["aa_boxes1"], g["aa_boxes2"], "box"), g["aa_expected"], atol=eps)
        assert np.allclose(oracle.box2d_iou(g["aa_boxes1"], g["aa_boxes2"], "rbox", alg=alg), g["aa_expected"], atol=4 * eps)
        assert np.allclose(oracle.box2d_iou(g["rot_boxes1"], g["rot_boxes2"], "box"), g["rot_box_expected"], atol=2 * eps)
        assert np.allclose(oracle.box2d_iou(g["rot_boxes1"], g["rot_boxes2"], "rbox", alg=alg), g["rot_rbox_expected"], atol=4 * eps)
        ab = g["apart_boxes"]
        assert np.allclose(oracle.box2d_iou(ab, ab, "box") - np.eye(4), 0, atol=1e-6)
        rb = g["apart_rboxes"]
        d = oracle.box2d_iou(rb, rb, "rbox", alg=alg) - np.eye(5)
        np.fill_diagonal(d, 0)
        assert np.allclose(d, 0, atol=1e-6)


def test_iou_degenerate_list(oracle):
    """SURVEY 8(c) D1-D13: RC restatement reproduces the reference's (wrong) answers bit for bit in
    fp64; the truth clip returns the geometric values."""
    g = golden("iou_degenerate.npz")
    for i, name in enumerate(g["names"]):
        a, b = g["boxes1"][i:i + 1], g["boxes2"][i:i + 1]
        rc = oracle.iou2dr(a, b, oracle.ALG_RC)[0, 0]
        assert rc == g["ref_f64"][i] or (np.isnan(rc) and np.isnan(g["ref_f64"][i])), name
        assert abs(oracle.iou2dr_truth(a, b)[0, 0] - g["truth"][i]) < 1e-15, name
    expect = dict(D1=1 / 3, D4=1 / 7, D5=1 / 3, D8=0.0, D9=0.0, D10=1.0, D11=1 / 16, D12=0.0, D13=0.0)
    for i, name in enumerate(g["names"]):
        if str(name) in expect:
            assert abs(g["truth"][i] - expect[str(name)]) < 1e-12, name


# ------------------------------------------------------------------ NMS
def test_nms_known_answer_and_fixtures(oracle):
    g = golden("nms.npz")
    for m in ("box", "rbox"):
        k = oracle.box2d_nms(g["test_boxes"], g["test_scores"], m)
        assert np.array_equal(k, g["test_expected"])
        assert np.array_equal(k, g[f"test_ref_{m}"])
    A, B, s = g["c1_boxes"], g["c1_boxes_b"], g["c1_scores"]
    k = oracle.box2d_nms(A, s, "rbox", iou_threshold=0.5)
    assert k.sum() == 673 and np.array_equal(k, _unpack(g["c1_keep_rbox"], 1000))
    assert np.array_equal(oracle.box2d_nms(B, s, "rbox", iou_threshold=0.5), _unpack(g["c1_keep_rbox_b"], 1000))
    assert np.array_equal(oracle.box2d_nms(A, s, "box", iou_threshold=0.5), _unpack(g["c1_keep_box"], 1000))
    assert np.array_equal(oracle.box2d_nms(A, s, "rbox", iou_threshold=0.3, score_threshold=0.2),
                          _unpack(g["c1_keep_rbox_thr03_s02"], 1000))
    P, ps = g["prop_boxes"], g["prop_scores"]
    assert np.array_equal(oracle.box2d_nms(P, ps, "rbox", iou_threshold=0.5), _unpack(g["prop_keep_rbox"], len(P)))
    assert np.array_equal(oracle.box2d_nms(P, ps, "box", iou_threshold=0.5), _unpack(g["prop_keep_box"], len(P)))
    # the truth clip gives the same fp64 decisions as RC on generic clustered proposals (SURVEY 8(c))
    assert np.array_equal(oracle.box2d_nms(P, ps, "rbox", iou_threshold=0.5, alg=oracle.ALG_TRUTH),
                          _unpack(g["prop_keep_rbox"], len(P)))


def test_nms_soft_smoke(oracle):
    """test/test_box.py:157-189: without a score threshold soft-NMS keeps everything."""
    boxes = np.array([[1, 1, 2, 2, 0], [2, 2, 2, 2, 0.01], [3, 3, 2, 2, 0.02], [3, 1, 1, 1, 0.03], [4, 2, 1, 1, 0.04],
                      [5, 3, 1, 1, 0.05]], np.float32)
    scores = np.array([0.5, 0.3, 0.4, 0.4, 0.2, 0.1], np.float32)
    for m in ("box", "rbox"):
        for s, p in (("linear", 1.0), ("gaussian", 0.5)):
            assert oracle.box2d_nms(boxes, scores, m, s, supression_param=p).all()


# ------------------------------------------------------------------ voxelization
def test_nms_soft_vs_reference_fixture(oracle):
    """LINEAR / GAUSSIAN suppression (f3): the oracle's restatement of nms.cpp:33-94 reproduces the keep masks written by the
    reference's own compiled CPU nms2d (tests/golden/make_golden.py write_soft_nms), fp64, bit for bit."""
    g = golden("nms_soft.npz")
    nb, ns = SOFT_TEST6
    for m, par in (("linear", 1.0), ("gaussian", 0.5)):
        for im in ("box", "rbox"):
            keep = oracle.box2d_nms(nb, ns, im, m, iou_threshold=0.1, score_threshold=0.15, supression_param=par)
            assert np.array_equal(keep, g[f"test6_{m}_{im}"]), (m, im)
    for tag, n, gen, m, it, st, par in SOFT_CASES:
        if n > 1000:
            continue   # the 4097-box cases take ~10 s each in the scalar oracle: covered by the GPU suite against the fixture
        b, s = soft_inputs(n, gen)
        im = "box" if tag.endswith("_box") else "rbox"
        keep = oracle.box2d_nms(b, s, im, m, iou_threshold=it, score_threshold=st, supression_param=par)
        assert np.array_equal(keep, np.unpackbits(g[tag])[:n].astype(bool)), tag


def test_voxel_spconv_golden(oracle):
    """test/test_voxel.py:80-88 + test/voxel_data.npz (spconv VoxelGeneratorV2 output)."""
    d = golden("voxel_spconv.npz")
    r = oracle.VoxelGenerator([0, 1, 0, 1, 0, 1], [10, 10, 10], max_points=5, max_points_filter="trim", dense=True)(d["cloud"])
    assert np.array_equal(r["voxels"], d["voxels"])
    assert np.array_equal(r["coords"], d["coords"])


def test_voxel_fixtures(oracle):
    g = golden("voxel_c2small.npz")
    pts = g["points"]
    cases = {
        "sp_default": dict(), "sp_trim5": dict(max_points=5, max_points_filter="trim"),
        "sp_trim2_v1000": dict(max_points=2, max_points_filter="trim", max_voxels=1000, max_voxels_filter="trim"),
        "sp_min2": dict(min_points=2, max_points=3, max_points_filter="trim"),
        "de_p5": dict(dense=True, max_points=5, max_voxels=20000), "de_p2_v1000": dict(dense=True, max_points=2, max_voxels=1000),
        "de_mean": dict(dense=True, max_points=3, max_voxels=20000, reduction="mean"),
        "de_max": dict(dense=True, max_points=3, max_voxels=20000, reduction="max"),
        "de_min": dict(dense=True, max_points=3, max_voxels=700, reduction="min"),
    }
    for name, kw in cases.items():
        r = oracle.VoxelGenerator(g["bounds"], g["shape"], **kw)(pts)
        _check_voxel(r, g, name, kw)
    for name, kw in {"co_trim5": dict(max_points=5, max_points_filter="trim"),
                     "co_de_mean": dict(dense=True, max_points=4, max_voxels=300, reduction="mean")}.items():
        r = oracle.VoxelGenerator(g["coarse_bounds"], g["coarse_shape"], **kw)(pts)
        _check_voxel(r, g, name, kw)


def _check_voxel(r, g, name, kw):
    for k, v in r.items():
        if k == "points":
            assert np.array_equal(v, g["points"][r["points_mask"]])
            continue
        exp = g[f"{name}.{k}"]
        if k == "voxel_pmask":  # reference leaves false slots uninitialised: compare the set slots only
            P = kw["max_points"]
            exp = np.unpackbits(exp)[:v.size].reshape(v.shape).astype(bool)
            sl = np.arange(P)[None, :] < np.minimum(r["voxel_npoints"], P)[:, None]
            assert np.array_equal(v[sl], exp[sl]) and v[sl].all() and not v[~sl].any(), (name, k)
        else:
            assert v.dtype == exp.dtype and np.array_equal(v, exp), (name, k)


def test_voxel_reference_properties(oracle):
    """test/test_voxel.py:11-78 semantic pins."""
    rng = np.random.default_rng(5)
    cloud = rng.random((2000, 4)).astype(np.float32)
    cloud = np.concatenate([cloud, np.array([[-1, -1, -1, -100], [-2, -2, -2, 100]], np.float32)])
    d = oracle.VoxelGenerator([0, 1, 0, 1, 0, 1], [10, 10, 10], reduction="mean", max_points=5, max_voxels=20000,
                              max_points_filter="trim", max_voxels_filter="trim", dense=True)(cloud)
    for i in range(len(d["voxels"])):
        for j in range(min(d["voxel_npoints"][i], 5)):
            assert (d["coords"][i] == (d["voxels"][i, j, :3] * np.float32(10)).astype(int)).all()
    s = oracle.VoxelGenerator([0, 1, 0, 1, 0, 1], [10, 10, 10])(cloud)
    assert len(s["points"]) == 2000 and len(s["coords"]) <= 1000
    assert (s["coords"][s["points_mapping"]] == (cloud[s["points_mask"], :3] * np.float32(10)).astype(int)).all()
    c3 = ((rng.random((2000, 3)) - 0.5) * 4).astype(np.float32)
    assert len(oracle.VoxelGenerator([0, 1, 0, 1, 0, 1], [10, 10, 10], max_voxels=10, max_voxels_filter="trim")(c3)["coords"]) <= 10
    assert len(oracle.VoxelGenerator([0, 1, 0, 1, 0, 1], [10, 10, 10], max_voxels=10, max_voxels_filter="descending")(c3)["coords"]) <= 10
    n = oracle.VoxelGenerator([-2, 2, -2, 2, -2, 2], [4, 4, 4], min_points=2, max_points=4, max_points_filter="trim")(c3)["voxel_npoints"]
    assert ((n >= 2) & (n <= 4)).all()


# ------------------------------------------------------------------ aligned scatter
def test_scatter_fixtures(oracle):
    g = golden("scatter.npz")
    for tag in ("f32", "f64"):
        for dim in (1, 2, 3):
            img, crd = g[f"{tag}.d{dim}.image"], g[f"{tag}.d{dim}.coord"]
            assert np.array_equal(oracle.scatter_forward(crd, img, 1), g[f"{tag}.d{dim}.mean"])
            assert np.array_equal(oracle.scatter_forward(crd, img, 2), g[f"{tag}.d{dim}.linear"])


def test_scatter_reference_known_answers(oracle):
    """test/test_point.py:10-69 (forward formulas and backward gradients)."""
    rng = np.random.default_rng(3)
    coord = np.array([[0, .25, .25, .25], [0, 1.25, 1.25, 1.25], [1, 2.25, 2.25, 2.25]], np.float32)
    img = rng.random((2, 10, 3, 3, 3)).astype(np.float32)
    m = oracle.scatter_forward(coord, img, 1)
    assert np.allclose(m[0], img[0, :, 0:2, 0:2, 0:2].reshape(10, -1).mean(1))
    assert np.allclose(m[1], img[0, :, 1:3, 1:3, 1:3].reshape(10, -1).mean(1))
    assert np.allclose(m[2], img[1, :, 2, 2, 2])
    lin = oracle.scatter_forward(coord, img, 2)
    w = np.array([.75, .25], np.float32)
    w3 = w[:, None, None] * w[None, :, None] * w[None, None, :]
    assert np.allclose(lin[0], (img[0, :, 0:2, 0:2, 0:2] * w3).reshape(10, -1).sum(1))
    assert np.allclose(lin[2], img[1, :, 2, 2, 2])
    ones = np.ones((3, 10), np.float32)
    gm = oracle.scatter_backward(coord, ones, 1, img.shape)
    assert np.allclose(gm[0, :, 0, 0, 0], 1 / 8) and np.allclose(gm[0, :, 1, 1, 1], 1 / 4) and np.allclose(gm[1, :, 2, 2, 2], 1)
    gl = oracle.scatter_backward(coord, ones, 2, img.shape)
    assert np.allclose(gl[0, :, 0, 0, 0], .75 ** 3) and np.allclose(gl[0, :, 1, 1, 1], .75 ** 3 + .25 ** 3)
    assert np.allclose(gl[1, :, 2, 2, 2], 1)
    # integral-coordinate quirk (SURVEY Appendix A): LINEAR doubles per integral in-range dim
    img2 = np.zeros((1, 1, 3, 3), np.float32); img2[0, 0, 1, 1] = 4.0; img2[0, 0, 2, 1] = 7.0
    assert oracle.scatter_forward(np.array([[0, 1.0, 1.0]], np.float32), img2, 2)[0, 0] == 16.0
    assert oracle.scatter_forward(np.array([[0, 1.5, 1.0]], np.float32), img2, 2)[0, 0] == 11.0
    assert oracle.scatter_forward(np.array([[0, 1.0, 1.0]], np.float32), img2, 1)[0, 0] == 4.0


# ------------------------------------------------------------------ the reference's own code: stored outputs, and live where oracle/_ref is built
def _live(part):
    """oracle.ref when the named part of the reference's compiled code is present (oracle/_ref is built from the reference source
    tree, which is not part of this repository), else None"""
    from oracle import ref as R
    try:
        getattr(R, part)()
    except OSError:
        return None
    return R


def test_oracle_vs_live_reference(oracle):
    """rotated / axis-aligned IoU, NMS with a score threshold and a 352x400x40 voxel grid with a voxel budget: the oracle against the
    outputs stored in tests/golden/live_ref.npz, and against the reference's extensions live where they are built"""
    g = golden("live_ref.npz")
    A, B, s, pts = live_iou_nms_voxel_inputs()
    bounds, shape, kw = LIVE_VOXEL
    assert_pinned(g, "rbox", oracle.iou2dr(A, B))
    assert_pinned(g, "box", oracle.iou2d(A, B))
    assert_pinned(g, "nms_keep", oracle.box2d_nms(A, s, "rbox", iou_threshold=0.4, score_threshold=0.1))
    a = oracle.VoxelGenerator(bounds, shape, **kw)(pts)
    assert sorted(a) == sorted(k[6:] for k in g.files if k.startswith("voxel."))
    for k in a:
        assert_pinned(g, "voxel." + k, a[k])
    from oracle import ref as R
    if not R.available():
        return
    assert np.array_equal(oracle.iou2dr(A, B), R.box2d_iou(A, B, "rbox"))
    assert np.array_equal(oracle.iou2d(A, B), R.box2d_iou(A, B, "box"))
    assert np.array_equal(oracle.box2d_nms(A, s, "rbox", iou_threshold=0.4, score_threshold=0.1),
                          R.box2d_nms(A, s, "rbox", iou_threshold=0.4, score_threshold=0.1))
    b = R.VoxelGenerator(bounds, shape, **kw)(pts)
    for k in b:
        assert np.array_equal(a[k], b[k]), k


def test_box3d_iou_distance_known_answers(oracle):
    """SURVEY 8(f) f1 (evaluator distance 1 - iou2d * ziou, d3d/dgal_wrap.h:45-91): z semantics of the restatement"""
    a = np.array([[0, 0, 0, 4, 2, 2, 0.3]], np.float32)
    cases = np.array([[0, 0, 0, 4, 2, 2, 0.3],      # identical -> 0
                      [0, 0, 5, 4, 2, 2, 0.3],      # disjoint in z -> 1
                      [0, 0, 1, 4, 2, 2, 0.3],      # same footprint, half z overlap: 1 - 1 * (1 / 3)
                      [0, 0, 0, 4, 2, 0, 0.3],      # flat box: i = 0
                      [50, 0, 0, 4, 2, 2, 0.3]], np.float32)
    for metric in ("riou", "iou"):
        d = oracle.box3d_iou_distance(a, cases, metric)
        assert d.dtype == np.float32 and np.allclose(d[0], [0, 1, 1 - 1 / 3, 1, 1], atol=1e-6)
    big = np.array([[0, 0, 0, 5000, 2, 2, 0.0]], np.float32)   # sizes are clipped to 1e3 (matcher.pyx:50-52)
    ref = np.array([[0, 0, 0, 1000, 2, 2, 0.0]], np.float32)
    assert np.allclose(oracle.box3d_iou_distance(big, ref, "iou"), 0, atol=1e-6)


def test_box3d_iou_distance_pinned(oracle):
    """f1: the restatement equals, bit for bit, the distances written by the reference's own box3dr_iou / box3d_iou (d3d/dgal_wrap.h
    compiled by g++: tests/golden/dist3d.npz and, on 150 x 120 more boxes, live_ref.npz) and that library live where oracle/_ref holds it"""
    g = golden("dist3d.npz")
    for metric in ("riou", "iou"):
        assert np.array_equal(oracle.box3d_iou_distance(g["src"], g["dst"], metric), g[metric]), metric
    g = golden("live_ref.npz")
    a, b, p3 = live_dist3d_inputs()
    for metric in ("riou", "iou"):
        assert_pinned(g, "dist3d." + metric, oracle.box3d_iou_distance(a, b, metric))
    # box3dr_pdist (d3d/dgal_wrap.h:21-43) against the tensor form of d3d/box/__init__.py:348-381 (fp32: equal up to hypot/sqrt rounding)
    pd = np.stack([oracle.box3dr_pdist(p3, a[k:k + 1])[0] for k in range(5)])
    assert np.abs(pd - g["box3dr_pdist"]).max() < 1e-5
    R = _live("_wrap")
    if R is None:
        return
    for metric in ("riou", "iou"):
        assert np.array_equal(oracle.box3d_iou_distance(a, b, metric), R.box3d_iou_distance(a, b, metric))
    for k in range(5):
        assert np.abs(pd[k] - R.box3dr_pdist_scalar(a[k], p3)).max() < 1e-5


def test_match_greedy_known_answers(oracle):
    """f1: ScoreMatcher.match restated (d3d/tracking/matcher.pyx:93-122, 138-162): best score first, closest free box of the same
    category within the threshold"""
    d = np.array([[0.2, 0.1, 0.9], [0.15, 0.3, 0.4], [0.5, 0.05, 0.1]], np.float32)
    sa, da = oracle.match_greedy(d, [0.9, 0.8, 0.7], [0, 0, 0], [0, 0, 0], [0.45])
    assert sa.tolist() == [1, 0, 2] and da.tolist() == [1, 0, 2]
    sa, da = oracle.match_greedy(d, [0.1, 0.8, 0.7], [0, 0, 0], [0, 0, 0], [0.45])     # source 1 first, then 2, then 0 (only box 2 left: 0.9 > thr)
    assert sa.tolist() == [-1, 0, 1] and da.tolist() == [1, 2, -1]
    sa, da = oracle.match_greedy(d, [0.9, 0.8, 0.7], [0, 1, 0], [1, 0, 0], [0.45, 0.2])  # categories: source 1 may only take box 0 (0.15 <= 0.2)
    assert sa.tolist() == [1, 0, 2] and da.tolist() == [1, 0, 2]
    sa, da = oracle.match_greedy(d, [0.9, 0.8, 0.7], [0, 1, 0], [1, 0, 0], [0.45, 0.1])
    assert sa.tolist() == [1, -1, 2]


def test_crop_2dr_pinned(oracle):
    """SURVEY 8(f) f4: point-in-rotated-box mask -- oracle == the reference's own crop_2dr (golden fixture, and the live
    extension when oracle/_ref exists) bit for bit, plus the known answers of reference test/test_box.py:191-205"""
    g = golden("crop.npz")
    for tag in ("f32", "f64"):
        pts, bx = g[f"{tag}.points"], g[f"{tag}.boxes"]
        exp = np.unpackbits(g[f"{tag}.mask"])[:len(bx) * len(pts)].reshape(len(bx), len(pts)).astype(bool)
        assert np.array_equal(oracle.crop_2dr(pts, bx), exp), tag
    rng = np.random.default_rng(3)
    cloud = (rng.random((100, 2)) * 2 - 1).astype(np.float32)
    boxes = np.array([[0, 0, 1, 1, 0], [0, 0, 1, 1, np.pi / 2 / 2]], np.float32)
    m = oracle.crop_2dr(cloud, boxes)
    ab = np.abs(cloud)
    assert np.array_equal(m[0], np.all(ab < 0.5, 1))
    assert np.array_equal(m[1], np.abs(ab[:, 0] + ab[:, 1]) < np.sqrt(2) / 2)
    p3 = np.concatenate([cloud, rng.normal(0, 1, (100, 1)).astype(np.float32)], 1)
    b3 = np.array([[0, 0, 0.2, 1, 1, 1.5, 0.3]], np.float32)
    m3 = oracle.box3dp_crop(p3, b3)
    assert m3.shape == (1, 100) and np.array_equal(m3[0], oracle.crop_2dr(p3[:, :2], b3[:, [0, 1, 3, 4, 6]])[0] & (np.abs(p3[:, 2] - 0.2) < 0.75))


def test_pdist2dr_pinned(oracle):
    """f4: the oracle's signed point-to-box distance equals, bit for bit in fp32 and fp64, the fixture written by the reference's own
    pdist2dr_forward (tests/golden/make_golden.py write_pdist) and the reference live when it is built; the point gradients of the
    reference's backward agree with central differences of the pinned forward."""
    g = golden("pdist.npz")
    for tag in ("f32", "f64"):
        d, ie = oracle.pdist2dr(g[f"{tag}.points"], g[f"{tag}.boxes"], return_iedge=True)
        assert d.dtype == g[f"{tag}.dist"].dtype and np.array_equal(d, g[f"{tag}.dist"]) and np.array_equal(ie, g[f"{tag}.iedge"]), tag
    pts, bx, up = g["f64.points"][:40], g["f64.boxes"], g["f64.grad"][:, :40]
    eps, num = 1e-6, np.zeros((40, 2))
    for j in range(40):
        for k in range(2):
            hi, lo = pts.copy(), pts.copy()
            hi[j, k] += eps; lo[j, k] -= eps
            num[j, k] = ((oracle.pdist2dr(hi, bx) - oracle.pdist2dr(lo, bx)) * up).sum() / (2 * eps)
    # the fixture's gradient sums over all 24 boxes for the same upstream gradient
    assert np.abs(num - g["f64.grad_points"][:40]).max() < 1e-6
    # 2000 points x 50 boxes: against the outputs stored in live_ref.npz, and the reference live where oracle/_ref holds it
    g = golden("live_ref.npz")
    pts, bx, p3, b3 = live_pdist_inputs()
    d, ie = oracle.pdist2dr(pts, bx, return_iedge=True)
    assert_pinned(g, "pdist2dr", d)
    assert_pinned(g, "pdist2dr.iedge", ie)
    assert oracle.box3dr_pdist(p3, b3).shape == (20, 500)
    R = _live("_box")
    if R is None:
        return
    rd, rie = R.pdist2dr(pts, bx)
    assert np.array_equal(d, rd) and np.array_equal(ie, rie)


def test_iou_ex_pinned(oracle):
    """f2: rotated GIoU / DIoU of the oracle (definitions over the pinned rotated IoU) against the values written by the reference's own
    giou2dr_forward / diou2dr_forward (tests/golden/make_golden.py write_iou_grad), and the fixture's gradients against central
    differences of the oracle on a few boxes: the fixture is a true gradient, so it can pin the CUDA backward"""
    g = golden("iou_grad.npz")
    A, B, up = g["boxes1"], g["boxes2"], g["grad"]
    for m in ("grbox", "drbox"):
        assert np.abs(oracle.iou2dr_ex(A, B, m) - g[m + ".value"]).max() < 1e-12, m
    assert np.abs(oracle.iou2dr_truth(A, B) - g["rbox.value"]).max() < 1e-12
    eps = 1e-6
    for m in ("grbox", "drbox"):
        for i in (0, 7):
            for k in range(5):
                hi, lo = A.copy(), A.copy()
                hi[i, k] += eps; lo[i, k] -= eps
                num = ((oracle.iou2dr_ex(hi[i:i + 1], B, m) - oracle.iou2dr_ex(lo[i:i + 1], B, m)) * up[i:i + 1]).sum() / (2 * eps)
                assert abs(num - g[m + ".grad1"][i, k]) < 1e-6, (m, i, k)
