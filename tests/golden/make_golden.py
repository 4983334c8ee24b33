"""Generate tests/golden/*.npz from the reference's OWN compiled CPU extensions (oracle/_ref).

Run in the authoring container, where /root/reference exists:
    python oracle/build_ref.py && python tests/golden/make_golden.py
The fixtures are small on purpose (the whole directory stays < 2 MB) and are what pins the C oracle
and the CUDA path on machines where the reference cannot be built (the GPU box has no /root/reference).
"""
import hashlib
import os
import shutil
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
OUT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(OUT))
from oracle import build_ref  # noqa: E402
from oracle import ref as R  # noqa: E402
from oracle import oracle as O  # noqa: E402
PI = np.pi


def gen_boxes(rng, n):
    """Reference benchmark distribution, test/compare/benchmark_riou.py:70-74 (SURVEY Appendix C)."""
    return np.stack([(rng.random(n) - .5) * 10, (rng.random(n) - .5) * 10, rng.random(n) * 5, rng.random(n) * 5,
                     (rng.random(n) - .5) * 10], 1)


def lidar(rng, n, rho_max=80.0, span=3.6):
    rho = rho_max * rng.random(n) ** 2
    th = (rng.random(n) - .5) * span
    z = rng.normal(-1.2, 0.6, n)
    inten = rng.random(n)
    return np.stack([rho * np.cos(th), rho * np.sin(th), z, inten], 1).astype(np.float32)


def proposals(rng, n, n_obj, extent=75.0):
    """Clustered BEV proposals (SURVEY 8(d) C3): centre + N(0,.3), size (4.5,2.0)+N(0,(.2,.1)), heading + N(0,.05)."""
    ctr = (rng.random((n_obj, 2)) - .5) * 2 * extent
    hd = (rng.random(n_obj) - .5) * 2 * PI
    k = rng.integers(0, n_obj, n)
    xy = ctr[k] + rng.normal(0, 0.3, (n, 2))
    wh = np.array([4.5, 2.0]) + rng.normal(0, 1, (n, 2)) * np.array([.2, .1])
    r = hd[k] + rng.normal(0, 0.05, n)
    scores = rng.permutation(n).astype(np.float64) / n + rng.random(n) * 0.1 / n  # distinct
    return np.concatenate([xy, wh, r[:, None]], 1), scores


def write_crop():
    """point-in-rotated-box masks of the reference's own crop_2dr (d3d/box/utils.cpp:10-47), bits packed"""
    rng = np.random.default_rng(9)
    out = {}
    for tag, dt in (("f32", np.float32), ("f64", np.float64)):
        pts = ((rng.random((3000, 2)) - .5) * 12).astype(dt)
        bx = gen_boxes(rng, 96).astype(dt)
        bx[:4] = np.array([[0, 0, 1, 1, 0], [0, 0, 1, 1, np.pi / 2], [0, 0, 0, 2, 0.3], [1, 1, 2, 2, 100.0]], dt)   # test_box.py:191-205 boxes, a flat box, a huge angle
        out[f"{tag}.points"], out[f"{tag}.boxes"] = pts, bx
        out[f"{tag}.mask"] = np.packbits(R.crop_2dr(pts, bx))
    np.savez_compressed(os.path.join(OUT, "crop.npz"), **out)


SOFT_CASES = [  # (tag, n, generator, method, iou_threshold, score_threshold, supression_param)
    ("c1_lin", 1000, "boxes", "linear", 0.3, 0.2, 1.0), ("c1_gau", 1000, "boxes", "gaussian", 0.3, 0.2, 0.5),
    ("c1_lin0", 1000, "boxes", "linear", 0.0, 0.0, 2.0), ("c1_gau_box", 1000, "boxes", "gaussian", 0.25, 0.3, 0.3),
    ("p_lin", 4097, "proposals", "linear", 0.3, 0.1, 1.0), ("p_gau", 4097, "proposals", "gaussian", 0.5, 0.05, 0.5),
]


def soft_inputs(n, gen):
    """inputs of the soft-NMS fixtures: regenerated from the seed by the tests, only the masks are stored"""
    rng = np.random.default_rng(1234 + n)
    if gen == "boxes":
        return gen_boxes(rng, n), rng.random(n)
    return proposals(rng, n, max(n // 25, 1))


def write_soft_nms():
    """keep masks of the reference's own CPU nms2d (d3d/box/nms.cpp:9-119) for the LINEAR / GAUSSIAN rules, fp64, bits packed"""
    nb = np.array([[1, 1, 2 - 1e-2, 2 - 1e-2, 0], [2, 2, 2 - 1e-2, 2 - 1e-2, 1e-3], [3, 3, 2 - 1e-2, 2 - 1e-2, 2e-3], [3, 1, 1, 2, 3e-3],
                   [4, 2, 1, 2, 4e-3], [5, 3, 1, 2, 5e-3]], np.float64)
    ns = np.array([0.5, 0.3, 0.4, 0.4, 0.2, 0.1], np.float64)
    out = {}
    for m, par in (("linear", 1.0), ("gaussian", 0.5)):
        for im in ("box", "rbox"):
            out[f"test6_{m}_{im}"] = R.box2d_nms(nb, ns, im, m, iou_threshold=0.1, score_threshold=0.15, supression_param=par)
    for tag, n, gen, m, it, st, par in SOFT_CASES:
        b, s = soft_inputs(n, gen)
        im = "box" if tag.endswith("_box") else "rbox"
        out[tag] = np.packbits(R.box2d_nms(b, s, im, m, iou_threshold=it, score_threshold=st, supression_param=par))
    np.savez_compressed(os.path.join(OUT, "nms_soft.npz"), **out)


def write_pdist():
    """signed point-to-box distances and edge indices of the reference's own pdist2dr_forward (d3d/box/dist.cpp:11-47), and the point
    gradients of its pdist2dr_backward for a fixed upstream gradient (its box gradients overwrite instead of accumulating,
    utils.h make_box_grad, and are not a reference for anything)"""
    rng = np.random.default_rng(11)
    out = {}
    for tag, dt in (("f32", np.float32), ("f64", np.float64)):
        pts = ((rng.random((300, 2)) - .5) * 12).astype(dt)
        bx = gen_boxes(rng, 24).astype(dt)
        bx[:3] = np.array([[0, 0, 1, 1, 0], [0, 0, 2, 1, np.pi / 2], [1, 1, 2, 2, 100.0]], dt)   # axis-aligned edges hit the b == 0 / a == 0 branches of t_from_pxy
        bx[:, 2:4] += 0.25
        d, ie = R.pdist2dr(pts, bx)
        g = rng.random(d.shape).astype(dt)
        gb, gp = R.pdist2dr_backward(pts, bx, g, ie)
        out[f"{tag}.points"], out[f"{tag}.boxes"], out[f"{tag}.dist"], out[f"{tag}.iedge"] = pts, bx, d, ie
        out[f"{tag}.grad"], out[f"{tag}.grad_points"] = g, gp
    np.savez_compressed(os.path.join(OUT, "pdist.npz"), **out)


def write_iou_grad():
    """values and gradients of the reference's own differentiable IoU family (d3d/box/iou.cpp:11-419, single-threaded), fp64"""
    rng = np.random.default_rng(33)
    A, B = gen_boxes(rng, 40), gen_boxes(rng, 30)
    A[:, 2:4] += 0.3; B[:, 2:4] += 0.3
    B[:6] = A[:6] + rng.normal(0, 0.2, (6, 5))       # strongly overlapping pairs
    up = rng.random((40, 30))
    out = dict(boxes1=A, boxes2=B, grad=up)
    for m in ("box", "rbox", "grbox", "drbox"):
        v, g1, g2 = R.iou_forward_backward(A, B, up, m)
        out[m + ".value"], out[m + ".grad1"], out[m + ".grad2"] = v, g1, g2
    np.savez_compressed(os.path.join(OUT, "iou_grad.npz"), **out)


def write_nms_c3():
    """keep mask of the reference's own CPU nms2d on the full C3 frame (50 000 clustered proposals, rbox, thr 0.5, fp64; ~25 s), bits packed"""
    P, ps = proposals(np.random.default_rng(2), 50000, 2000)
    np.savez_compressed(os.path.join(OUT, "nms_c3.npz"), keep=np.packbits(R.box2d_nms(P, ps, "rbox", iou_threshold=0.5)))


def write_dist3d():
    """detection-evaluation distances 1 - iou2d * ziou of the reference's own box3dr_iou / box3d_iou (d3d/dgal_wrap.h:45-91, g++)"""
    rng = np.random.default_rng(21)

    def b3(n):
        return np.concatenate([(rng.random((n, 2)) - .5) * 10, rng.normal(0, 0.5, (n, 1)), rng.random((n, 3)) * 4 + .3,
                               (rng.random((n, 1)) - .5) * 10], 1).astype(np.float32)
    a, b = b3(60), b3(45)
    b[:5] = a[:5]                      # identical boxes
    b[5, 2] += 50                      # no z overlap
    np.savez_compressed(os.path.join(OUT, "dist3d.npz"), src=a, dst=b, riou=R.box3d_iou_distance(a, b, "riou"), iou=R.box3d_iou_distance(a, b, "iou"))


def pin(out, name, a, sample=1024):
    """store a large array for conftest.assert_pinned: the SHA-256 of its bytes, its shape and its values at a fixed sample of positions"""
    a = np.ascontiguousarray(a)
    idx = np.sort(np.random.default_rng(0).choice(a.size, min(sample, a.size), replace=False))
    out[name + ".sha256"] = np.array(hashlib.sha256(a.tobytes()).hexdigest())
    out[name + ".shape"] = np.array(a.shape, np.int64)
    out[name + ".idx"], out[name + ".val"] = idx, a.reshape(-1)[idx]


def write_live_ref():
    """outputs on the inputs of the comparisons of tests/test_oracle_pinned.py with the reference's own code (conftest live_*_inputs):
    rotated / axis-aligned IoU, NMS and voxelization (box_impl, voxel_impl), evaluator distances and box3dr_pdist (dgal_wrap.h),
    pdist2dr_forward (box_impl).  They come from the reference where oracle/_ref is built; elsewhere from the oracle, which then pins the
    oracle on these inputs to the values it had when the file was written.  `source` records which of the two wrote the file."""
    from conftest import LIVE_VOXEL, live_dist3d_inputs, live_iou_nms_voxel_inputs, live_pdist_inputs
    ref = R.available() and os.path.exists(build_ref.WRAP_SO)
    out = dict(source=np.array("reference" if ref else "oracle"))
    A, B, s, pts = live_iou_nms_voxel_inputs()
    pin(out, "rbox", R.box2d_iou(A, B, "rbox") if ref else O.iou2dr(A, B))
    pin(out, "box", R.box2d_iou(A, B, "box") if ref else O.iou2d(A, B))
    out["nms_keep"] = (R.box2d_nms if ref else O.box2d_nms)(A, s, "rbox", iou_threshold=0.4, score_threshold=0.1)
    bounds, shape, kw = LIVE_VOXEL
    for k, v in (R if ref else O).VoxelGenerator(bounds, shape, **kw)(pts).items():
        out["voxel." + k] = v
    a, b, p3 = live_dist3d_inputs()
    for metric in ("riou", "iou"):
        out["dist3d." + metric] = (R if ref else O).box3d_iou_distance(a, b, metric)
    out["box3dr_pdist"] = np.stack([R.box3dr_pdist_scalar(a[k], p3) if ref else O.box3dr_pdist(p3, a[k:k + 1])[0] for k in range(5)])
    pts, bx, _, _ = live_pdist_inputs()
    d, ie = R.pdist2dr(pts, bx) if ref else O.pdist2dr(pts, bx, return_iedge=True)
    pin(out, "pdist2dr", d)
    out["pdist2dr.iedge"] = ie
    np.savez_compressed(os.path.join(OUT, "live_ref.npz"), **out)


def main():
    assert R.available(), "build oracle/_ref first"
    if "--only-crop" in sys.argv:
        return write_crop()
    # ---------------- IoU: C1-style random, 160x96 block (fp64 + fp32, rbox + box)
    rng = np.random.default_rng(0)
    A, B = gen_boxes(rng, 1000), gen_boxes(rng, 1000)
    scores = rng.random(1000)
    a, b = A[:160], B[:96]
    np.savez_compressed(
        os.path.join(OUT, "iou_c1.npz"), boxes1=a, boxes2=b,
        rbox_f64=R.box2d_iou(a, b, "rbox"), box_f64=R.box2d_iou(a, b, "box"),
        rbox_f32=R.box2d_iou(a.astype(np.float32), b.astype(np.float32), "rbox", precise=False),
        box_f32=R.box2d_iou(a.astype(np.float32), b.astype(np.float32), "box", precise=False),
        # whole-matrix anchors of config C1 (SURVEY Appendix C)
        c1_rbox_sum=R.box2d_iou(A, B, "rbox").sum(), c1_rbox_nnz=(R.box2d_iou(A, B, "rbox") != 0).sum(),
        c1_box_sum=R.box2d_iou(A, B, "box").sum())

    # ---------------- IoU: degenerate list D1..D13 (SURVEY 8(c)); ref fp64 / fp32 and truth
    s2 = np.sqrt(2.0)
    D = [
        ("D1", (0, 0, 2, 2, .1), (np.cos(.1), np.sin(.1), 2, 2, .1)),
        ("D2", (0, 0, 4, 2, .7), (.5, .3, 4, 2, .7)),
        ("D3", (0, 0, 4, 2, .3), (.5, .3, 3, 1.5, .3)),
        ("D4", (0, 0, 2, 2, 0), (1, 1, 2, 2, 0)),
        ("D5", (0, 0, 4, 2, .3), (.5, .3, 4, 2, .3 + PI / 2)),
        ("D6", (0, 0, 4, 2, .3), (.5, .3, 4, 2, .3 + PI)),
        ("D7", (0, 0, 4, 2, .3), (.5, .3, 4, 2, .3 + 1e-9)),
        ("D8", (0, 0, 2, 2, 0), (2, 0, 2, 2, 0)),
        ("D9", (0, 0, 2, 2, 0), (2, 2, 2 * s2, 2 * s2, PI / 4)),
        ("D10", (1.5, -2, 3, 1, .77), (1.5, -2, 3, 1, .77)),
        ("D11", (0, 0, 4, 4, .1), (0, 0, 1, 1, .5)),
        ("D12", (0, 0, 0, 2, .2), (0, 0, 2, 2, .1)),
        ("D13", (0, 0, 2, 2, .3), (50, 50, 2, 2, 1.3)),
    ]
    d1 = np.array([d[1] for d in D], np.float64)
    d2 = np.array([d[2] for d in D], np.float64)
    ref64 = np.array([R.box2d_iou(d1[i:i + 1], d2[i:i + 1], "rbox")[0, 0] for i in range(len(D))])
    ref32 = np.array([R.box2d_iou(d1[i:i + 1].astype(np.float32), d2[i:i + 1].astype(np.float32), "rbox",
                                  precise=False)[0, 0] for i in range(len(D))])
    truth = np.array([O.iou2dr_truth(d1[i:i + 1], d2[i:i + 1])[0, 0] for i in range(len(D))])
    np.savez_compressed(os.path.join(OUT, "iou_degenerate.npz"), names=np.array([d[0] for d in D]), boxes1=d1,
                        boxes2=d2, ref_f64=ref64, ref_f32=ref32, truth=truth)

    # ---------------- IoU: the reference's own known-answer tests (test/test_box.py:12-100)
    eps = 1e-3
    d90 = PI / 4
    np.savez_compressed(
        os.path.join(OUT, "iou_known_answers.npz"),
        aa_boxes1=np.array([[1, 1, 2, 2, eps], [2, 2, 2, 2, eps], [3, 3, 2, 2, eps]], np.float32),
        aa_boxes2=np.array([[3, 1, 2, 2, -eps], [2, 2, 2, 2, -eps], [1, 3, 2, 2, -eps]], np.float32),
        aa_expected=np.array([[0, 1 / 7, 0], [1 / 7, 1, 1 / 7], [0, 1 / 7, 0]], np.float32),
        rot_boxes1=np.array([[0, 0, 2, 2, 0], [-1, 1, 2, 2, 0], [1, 1, 2, 2, 0]], np.float32),
        rot_boxes2=np.array([[-1, 1, 2 * s2 - eps, 2 * s2 - eps, d90 - eps], [1, 1, s2 + eps, s2 + eps, d90 + eps]],
                            np.float32),
        rot_box_expected=np.array([[1 / 4, 1 / 7], [1 / 4, 0], [1 / 9, 1]], np.float32),
        rot_rbox_expected=np.array([[1 / 5, 1 / 11], [1 / 2, 0], [1 / 11, 1 / 2]], np.float32),
        apart_boxes=np.array([[1, 2, 3, 3, 0], [-2, 1, 3, 3, 0], [-1, -2, 3, 3, 0], [2, -1, 3, 3, 0]], np.float32),
        apart_rboxes=np.array([[0, 0, 2, 2, 0], [2, 2, 2 * s2, 2 * s2, d90 + eps], [-2, 2, 2 * s2, 2 * s2, d90 + 2 * eps],
                               [2, -2, 2 * s2, 2 * s2, d90 + 3 * eps], [-2, -2, 2 * s2, 2 * s2, d90 + 4 * eps]],
                              np.float32))

    # ---------------- NMS
    nb = np.array([[1, 1, 2 - 10 * eps, 2 - 10 * eps, 0], [2, 2, 2 - 10 * eps, 2 - 10 * eps, eps],
                   [3, 3, 2 - 10 * eps, 2 - 10 * eps, 2 * eps], [3, 1, 1, 2, 3 * eps], [4, 2, 1, 2, 4 * eps],
                   [5, 3, 1, 2, 5 * eps]], np.float32)
    ns = np.array([0.5, 0.3, 0.4, 0.4, 0.2, 0.1], np.float32)
    rng3 = np.random.default_rng(2)
    P, ps = proposals(rng3, 3000, 120)
    out = dict(test_boxes=nb, test_scores=ns, test_expected=np.array([1, 0, 1, 1, 0, 1], bool),
               test_ref_box=R.box2d_nms(nb, ns, "box"), test_ref_rbox=R.box2d_nms(nb, ns, "rbox"),
               c1_boxes=A, c1_boxes_b=B, c1_scores=scores,
               c1_keep_rbox=np.packbits(R.box2d_nms(A, scores, "rbox", iou_threshold=0.5)),
               c1_keep_rbox_b=np.packbits(R.box2d_nms(B, scores, "rbox", iou_threshold=0.5)),
               c1_keep_box=np.packbits(R.box2d_nms(A, scores, "box", iou_threshold=0.5)),
               c1_keep_rbox_thr03_s02=np.packbits(R.box2d_nms(A, scores, "rbox", iou_threshold=0.3, score_threshold=0.2)),
               prop_boxes=P, prop_scores=ps,
               prop_keep_rbox=np.packbits(R.box2d_nms(P, ps, "rbox", iou_threshold=0.5)),
               prop_keep_box=np.packbits(R.box2d_nms(P, ps, "box", iou_threshold=0.5)),
               prop_keep_rbox_f32=np.packbits(R.box2d_nms(P.astype(np.float32), ps.astype(np.float32), "rbox",
                                                          iou_threshold=0.5, precise=False)))
    np.savez_compressed(os.path.join(OUT, "nms.npz"), **out)

    # ---------------- voxelization: the reference's spconv golden + a C2-shaped 6000-point cloud
    shutil.copyfile(os.path.join(os.environ.get("D3D_REFERENCE_ROOT", "/root/reference"), "test", "voxel_data.npz"),
                    os.path.join(OUT, "voxel_spconv.npz"))
    rng1 = np.random.default_rng(1)
    pts = lidar(rng1, 6000)
    pts[:40, :3] = pts[40:80, :3]  # duplicates -> multi-point voxels
    pts[100:140, :3] = pts[40:80, :3] + np.float32(1e-3)
    bounds, shape = [0, 70.4, -40, 40, -3, 1], [1408, 1600, 40]
    vox = dict(points=pts, bounds=np.array(bounds, np.float32), shape=np.array(shape, np.int32))
    cases = {
        "sp_default": dict(),
        "sp_trim5": dict(max_points=5, max_points_filter="trim"),
        "sp_trim2_v1000": dict(max_points=2, max_points_filter="trim", max_voxels=1000, max_voxels_filter="trim"),
        "sp_min2": dict(min_points=2, max_points=3, max_points_filter="trim"),
        "de_p5": dict(dense=True, max_points=5, max_voxels=20000),
        "de_p2_v1000": dict(dense=True, max_points=2, max_voxels=1000),
        "de_mean": dict(dense=True, max_points=3, max_voxels=20000, reduction="mean"),
        "de_max": dict(dense=True, max_points=3, max_voxels=20000, reduction="max"),
        "de_min": dict(dense=True, max_points=3, max_voxels=700, reduction="min"),
    }
    for name, kw in cases.items():
        r = R.VoxelGenerator(bounds, shape, **kw)(pts)
        for k, v in r.items():
            if k == "points":
                continue  # == pts[points_mask]
            if k == "voxels":
                v = v.astype(np.float32)
            vox[f"{name}.{k}"] = np.packbits(v) if v.dtype == bool else v
    # coarse grid -> many points per voxel (exercises trimming and ordered sums)
    bounds2, shape2 = [0, 70.4, -40, 40, -3, 1], [44, 50, 4]
    for name, kw in {"co_trim5": dict(max_points=5, max_points_filter="trim"),
                     "co_de_mean": dict(dense=True, max_points=4, max_voxels=300, reduction="mean"),
                     "co_desc": dict(max_voxels=50, max_voxels_filter="descending", min_points=3)}.items():
        r = R.VoxelGenerator(bounds2, shape2, **kw)(pts)
        for k, v in r.items():
            if k == "points":
                continue
            vox[f"{name}.{k}"] = np.packbits(v) if v.dtype == bool else v
    vox["coarse_bounds"] = np.array(bounds2, np.float32)
    vox["coarse_shape"] = np.array(shape2, np.int32)
    np.savez_compressed(os.path.join(OUT, "voxel_c2small.npz"), **vox)

    # ---------------- aligned scatter: reference test case + random cases (forward from the reference;
    # backward expectations are the reference TEST's known answers, test/test_point.py:43-60, because the
    # reference CPU backward entry point never invokes its dispatch lambda (d3d/point/scatter.cpp:193-200)
    # and returns zeros at this commit)
    g = np.random.default_rng(7)
    sc = {}
    for dt, tag in ((np.float32, "f32"), (np.float64, "f64")):
        for dim, shp in ((1, (2, 5, 9)), (2, (2, 6, 7, 8)), (3, (2, 5, 4, 5, 6))):
            img = g.random(shp).astype(dt)
            n = 64
            crd = np.concatenate([g.integers(0, 2, (n, 1)).astype(dt),
                                  (g.random((n, dim)) * np.array(shp[2:]) * 1.3 - 1).astype(dt)], 1)
            crd[:12, 1:] = np.round(crd[:12, 1:])  # integral coordinates (reference doubles the weights)
            sc[f"{tag}.d{dim}.image"] = img
            sc[f"{tag}.d{dim}.coord"] = crd
            for meth in ("mean", "linear"):
                sc[f"{tag}.d{dim}.{meth}"] = R.aligned_scatter_forward(crd, img, meth)
    np.savez_compressed(os.path.join(OUT, "scatter.npz"), **sc)
    write_crop()
    write_live_ref()
    tot = sum(os.path.getsize(os.path.join(OUT, f)) for f in os.listdir(OUT) if f.endswith(".npz"))
    print("golden fixtures written, total bytes:", tot)


if __name__ == "__main__" and len(sys.argv) > 1:   # python make_golden.py soft_nms ...: only the named fixtures
    for name in sys.argv[1:]:
        globals()["write_" + name]()
elif __name__ == "__main__":
    main()
