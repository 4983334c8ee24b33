"""numpy front end of the CPU oracle (oracle/libd3d_oracle.so).  TEST INFRASTRUCTURE ONLY.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / `--impl reference` legs may import
this module; the product package d3d_b200/ never does (tests/test_no_oracle_in_product.py enforces it).

Each function mirrors one reference entry point (file:line in the docstring) and takes/returns numpy
arrays with the reference's layouts and dtypes.
"""
import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None

ALG_RC, ALG_SH, ALG_TRUTH = 1, 2, 3
IOU_BOX, IOU_RBOX = 1, 2
SUP_HARD, SUP_LINEAR, SUP_GAUSSIAN = 0, 1, 2


def build():
    subprocess.check_call(["make", "-s", "-C", HERE])


def lib():
    global _LIB
    if _LIB is None:
        p = os.path.join(HERE, "libd3d_oracle.so")
        if not os.path.exists(p):
            build()
        _LIB = C.CDLL(p)
        _LIB.orc_nms2d_f.restype = C.c_int64
        _LIB.orc_nms2d_d.restype = C.c_int64
        _LIB.orc_voxelize_dense.restype = C.c_int64
        _LIB.orc_voxelize_sparse.restype = C.c_int64
        _LIB.orc_voxelize_filter.restype = C.c_int64
    return _LIB


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def _boxes(b, dt):
    b = np.ascontiguousarray(b, dtype=dt)
    assert b.ndim == 2 and b.shape[1] == 5
    return b


def iou2dr(b1, b2, alg=ALG_RC, return_blowups=False):
    """Pairwise rotated IoU, dtype = b1.dtype (f32 or f64): reference d3d/box/iou.cpp:94-141."""
    dt = np.float32 if b1.dtype == np.float32 else np.float64
    b1, b2 = _boxes(b1, dt), _boxes(b2, dt)
    out = np.empty((len(b1), len(b2)), dt)
    bl = np.zeros(out.shape, np.uint8)
    f = lib().orc_iou2dr_f32 if dt == np.float32 else lib().orc_iou2dr_f64
    f(_p(b1), C.c_int64(len(b1)), _p(b2), C.c_int64(len(b2)), _p(out), C.c_int(alg), _p(bl))
    return (out, bl) if return_blowups else out


def iou2dr_truth(b1, b2):
    """Geometric truth (long-double closed half-plane clip) from float64 inputs."""
    b1, b2 = _boxes(b1, np.float64), _boxes(b2, np.float64)
    out = np.empty((len(b1), len(b2)), np.float64)
    lib().orc_iou2dr_truth(_p(b1), C.c_int64(len(b1)), _p(b2), C.c_int64(len(b2)), _p(out))
    return out


def iou2d(b1, b2):
    """Pairwise IoU of the AABBs of the rotated boxes (method="box"): d3d/box/iou.cpp:11-46."""
    dt = np.float32 if b1.dtype == np.float32 else np.float64
    b1, b2 = _boxes(b1, dt), _boxes(b2, dt)
    out = np.empty((len(b1), len(b2)), dt)
    f = lib().orc_iou2d_f32 if dt == np.float32 else lib().orc_iou2d_f64
    f(_p(b1), C.c_int64(len(b1)), _p(b2), C.c_int64(len(b2)), _p(out))
    return out


def box2d_iou(b1, b2, method="box", precise=True, alg=ALG_RC):
    """Front door: d3d/box/__init__.py:180-224 (dtype policy: fp64 compute when precise)."""
    otype = b1.dtype
    if precise:
        b1, b2 = b1.astype(np.float64), b2.astype(np.float64)
    r = iou2d(b1, b2) if method == "box" else iou2dr(b1, b2, alg)
    return r.astype(otype) if precise else r


def crop_2dr(points, boxes):
    """Point-in-rotated-box mask bool[M boxes, N points]: reference d3d/box/utils.cpp:10-47 (bound as crop_2dr,
    front door box2dr_crop d3d/box/__init__.py:278-287)."""
    dt = np.float32 if points.dtype == np.float32 else np.float64
    pts, bx = np.ascontiguousarray(points, dtype=dt), _boxes(boxes, dt)
    assert pts.ndim == 2 and pts.shape[1] == 2
    out = np.empty((len(bx), len(pts)), np.uint8)
    f = lib().orc_crop2dr_f32 if dt == np.float32 else lib().orc_crop2dr_f64
    f(_p(pts), C.c_int64(len(pts)), _p(bx), C.c_int64(len(bx)), _p(out))
    return out.astype(bool)


def pdist2dr(points, boxes, return_iedge=False):
    """Signed point-to-rotated-box distance T[M boxes, N points] (positive inside) and the edge that realises it: reference
    d3d/box/dist.cpp:11-47 pdist2dr_forward over dgal::distance (geometry.hpp:453-497)."""
    dt = np.float32 if points.dtype == np.float32 else np.float64
    pts = np.ascontiguousarray(points, dt)
    bx = _boxes(boxes, dt)
    dist = np.empty((len(bx), len(pts)), dt)
    ie = np.empty((len(bx), len(pts)), np.uint8)
    f = lib().orc_pdist2dr_f32 if dt == np.float32 else lib().orc_pdist2dr_f64
    f(_p(pts), C.c_int64(len(pts)), _p(bx), C.c_int64(len(bx)), _p(dist), _p(ie))
    return (dist, ie) if return_iedge else dist


def box3dr_pdist(points, boxes, project_axis=2):
    """d3d/box/__init__.py:344-381 with every term in the native [M boxes, N points] layout (the reference's wrapper hands
    (boxes, points) to a native function declared (points, boxes), d3d/box/__init__.py:151-153 against dist.h:7-9, and cannot run)."""
    ax2 = {0: ([1, 2], [1, 2, 4, 5, 6]), 1: ([0, 2], [0, 2, 3, 5, 6]), 2: ([0, 1], [0, 1, 3, 4, 6])}[project_axis]
    d2 = pdist2dr(np.ascontiguousarray(points[:, ax2[0]]), np.ascontiguousarray(boxes[:, ax2[1]]))
    pp = points[:, project_axis][None, :]
    ctr, half = boxes[:, project_axis][:, None], boxes[:, 3 + project_axis][:, None] / 2
    dp = np.where(pp > ctr, (ctr + half) - pp, pp - (ctr - half))
    return np.where(dp > 0, np.where(d2 > 0, np.minimum(dp, d2), d2), np.where(d2 > 0, dp, -np.sqrt(d2 * d2 + dp * dp))).astype(d2.dtype)


def _pdist_frame(dx, dy, w, h, r, return_iedge=False):
    """signed distance (positive inside) of the local offsets (dx, dy) = point - centre to the closed rectangle of half extents
    |w| / 2, |h| / 2 turned by r, all float64 arrays that broadcast.  The offset is turned into the box's frame; the magnitude is the
    least distance to its four edges as segments between the corners of pd_quad's order, (-w/2, -h/2), (w/2, -h/2), (w/2, h/2),
    (-w/2, h/2); the sign comes from the containment test.  The edge index is the first minimum in the loop order 3, 0, 1, 2."""
    c, s = np.cos(r), np.sin(r)
    qx, qy = c * dx + s * dy, c * dy - s * dx
    vx = [-w / 2, w / 2, w / 2, -w / 2]
    vy = [-h / 2, -h / 2, h / 2, h / 2]
    seg = []
    for k in range(4):   # edge k: v_k -> v_k+1
        ax, ay, bx, by = vx[k], vy[k], vx[(k + 1) % 4], vy[(k + 1) % 4]
        ex, ey = bx - ax, by - ay
        ll = ex * ex + ey * ey
        with np.errstate(invalid="ignore", divide="ignore"):
            t = np.where(ll > 0, np.clip(((qx - ax) * ex + (qy - ay) * ey) / np.where(ll > 0, ll, 1), 0, 1), 0)
        cx, cy = np.where(t >= 1, bx, ax + t * ex), np.where(t >= 1, by, ay + t * ey)   # the corners exactly: ties at corners stay ties
        seg.append(np.hypot(qx - cx, qy - cy))
    order = (3, 0, 1, 2)
    allseg = np.stack([seg[k] for k in order])
    dmin = allseg.min(0)
    inside = (np.abs(qx) <= np.abs(w) / 2) & (np.abs(qy) <= np.abs(h) / 2)
    d = np.where(inside, dmin, -dmin)
    if return_iedge:
        return d, np.asarray(order, np.uint8)[allseg.argmin(0)]
    return d


def pdist2dr_local(points, boxes, return_iedge=False):
    """Signed point-to-rotated-box distance T[M boxes, N points] (positive inside, zero on the boundary) in float64 with each pair moved
    into its box's frame: p - c is taken in float64 (exact for widened float32 inputs, and for float64 points near their box) and turned
    by -r.  The geometric truth that box2dr_pdist computes; pdist2dr above restates the reference, which differs from it on the lines
    through edges, at headings of pi / 2 and far from the origin (SURVEY.md 8(c), P1).  With return_iedge, also the index k of the edge
    v_k -> v_k+1 that realises the distance (ties: first of 3, 0, 1, 2)."""
    p, b = np.asarray(points, np.float64), np.asarray(boxes, np.float64)
    col = lambda k: b[:, k:k + 1]  # noqa: E731
    return _pdist_frame(p[None, :, 0] - col(0), p[None, :, 1] - col(1), col(2), col(3), col(4), return_iedge)


def pdist2dr_grad_local(points, boxes, h=1e-4, smooth_tol=1e-9):
    """Per-pair derivatives of pdist2dr_local by five-point differences, taken in the box's frame: returns (value [M, N],
    dp [M, N, 2] = d value / d points[j], db [M, N, 5] = d value / d boxes[i], smooth bool [M, N]).  A pair is smooth when the stencils at
    h and h / 2 agree to `smooth_tol` in all seven derivatives; elsewhere (a tie between two edges inside, the boundary, a zero extent)
    the value has a kink within the stencil and no derivative to compare with."""
    p, b = np.asarray(points, np.float64), np.asarray(boxes, np.float64)
    m, n = len(b), len(p)
    dx, dy = p[None, :, 0] - b[:, 0:1], p[None, :, 1] - b[:, 1:2]
    base = [dx, dy, np.zeros((m, 1)), np.zeros((m, 1)), b[:, 2:3], b[:, 3:4], b[:, 4:5]]   # point x, y, box x, y, w, h, r

    def f(args):
        return _pdist_frame(args[0] - args[2], args[1] - args[3], args[4], args[5], args[6])

    val = f(base)
    der, smooth = np.empty((m, n, 7)), np.ones((m, n), bool)
    for k in range(7):
        est = []
        for hh in (h, h / 2):
            fs = []
            for s in (-2, -1, 1, 2):
                a = list(base)
                a[k] = a[k] + s * hh
                fs.append(f(a))
            est.append((fs[0] - 8 * fs[1] + 8 * fs[2] - fs[3]) / (12 * hh))
        der[..., k] = est[0]
        smooth &= np.abs(est[0] - est[1]) <= smooth_tol
    return val, der[..., :2], der[..., 2:], smooth


def box3dr_pdist_local(points, boxes, project_axis=2):
    """box3dr_pdist in float64 from the local 2-D term (pdist2dr_local) and the signed distance along the projection axis: the signed
    distance to the boundary of the prism, positive inside."""
    p, b = np.asarray(points, np.float64), np.asarray(boxes, np.float64)
    ax2 = {0: ([1, 2], [1, 2, 4, 5, 6]), 1: ([0, 2], [0, 2, 3, 5, 6]), 2: ([0, 1], [0, 1, 3, 4, 6])}[project_axis]
    d2 = pdist2dr_local(p[:, ax2[0]], b[:, ax2[1]])
    dp = np.abs(b[:, 3 + project_axis])[:, None] / 2 - np.abs(p[None, :, project_axis] - b[:, project_axis][:, None])
    return np.where(dp > 0, np.where(d2 > 0, np.minimum(dp, d2), d2), np.where(d2 > 0, dp, -np.hypot(d2, dp)))


def box3dp_crop(points, boxes, project_axis=2):
    """d3d/box/__init__.py:289-314: 2-D crop of the projection & the open interval test along the projection axis."""
    ax2 = {0: ([1, 2], [1, 2, 4, 5, 6]), 1: ([0, 2], [0, 2, 3, 5, 6]), 2: ([0, 1], [0, 1, 3, 4, 6])}[project_axis]
    m2 = crop_2dr(np.ascontiguousarray(points[:, ax2[0]]), np.ascontiguousarray(boxes[:, ax2[1]]))
    pp, bp, bd = points[:, [project_axis]].T, boxes[:, [project_axis]], boxes[:, [3 + project_axis]] / 2
    return m2 & ((pp - bd < bp) & (bp < pp + bd))


def box3d_iou_distance(src, dst, metric="riou", alg=ALG_RC):
    """Distance cache of ScoreMatcher.prepare_boxes: 1 - iou2d * ziou in float32 for [N,7] / [M,7] boxes
    (x, y, z, lx, ly, lz, rz): reference d3d/tracking/matcher.pyx:45-76 over box3dr_iou / box3d_iou,
    d3d/dgal_wrap.h:45-91.  The BEV IoU comes from the pinned fp32 restatement above (alg: the reference's RC, or
    ALG_TRUTH for geometric truth); the z factor follows dgal_wrap.h:50-66 operation by operation in float32.
    PINNED: equal bit for bit to the reference's own box3dr_iou / box3d_iou (d3d/dgal_wrap.h compiled by g++ into
    oracle/_ref/libdgal_wrap.so through oracle/dgal_wrap_shim.cpp) live and on tests/golden/dist3d.npz."""
    f = np.float32
    a, b = np.array(src, dtype=f, copy=True), np.array(dst, dtype=f, copy=True)
    a[:, 3:6] = np.clip(a[:, 3:6], -1e3, 1e3)          # matcher.pyx:50-52
    b[:, 3:6] = np.clip(b[:, 3:6], -1e3, 1e3)
    a2, b2 = a[:, [0, 1, 3, 4, 6]], b[:, [0, 1, 3, 4, 6]]
    if metric == "riou":
        iou = iou2dr_truth(a2.astype(np.float64), b2.astype(np.float64)).astype(f) if alg == ALG_TRUTH else iou2dr(a2, b2, alg)
    else:
        iou = iou2d(a2, b2)
    z1max, z1min = (a[:, 2] + a[:, 5] / f(2))[:, None], (a[:, 2] - a[:, 5] / f(2))[:, None]
    z2max, z2min = (b[:, 2] + b[:, 5] / f(2))[None, :], (b[:, 2] - b[:, 5] / f(2))[None, :]
    i = np.maximum(np.minimum(z1max, z2max) - np.maximum(z1min, z2min), f(0))
    u = np.maximum(np.maximum(z1max, z2max) - np.minimum(z1min, z2min), f(1e-6))
    return (f(1) - iou.astype(f) * (i / u).astype(f)).astype(f)


def _hull_area_and_diameter(pts):
    """area of the convex hull (Andrew's monotone chain) and largest pairwise distance of a few points, float64"""
    p = sorted(map(tuple, pts))
    def half(seq):
        h = []
        for q in seq:
            while len(h) >= 2 and (h[-1][0] - h[-2][0]) * (q[1] - h[-2][1]) - (h[-1][1] - h[-2][1]) * (q[0] - h[-2][0]) <= 0:
                h.pop()
            h.append(q)
        return h
    hull = half(p)[:-1] + half(p[::-1])[:-1]
    area = 0.5 * abs(sum(hull[i][0] * hull[(i + 1) % len(hull)][1] - hull[i][1] * hull[(i + 1) % len(hull)][0] for i in range(len(hull))))
    pa = np.asarray(pts)
    diam = np.sqrt(((pa[:, None, :] - pa[None, :, :]) ** 2).sum(-1)).max()
    return area, diam


def iou2dr_ex(boxes1, boxes2, method="grbox"):
    """Rotated GIoU / DIoU [N, M] in float64 from their definitions (dgal::giou / diou, geometry.hpp:1241-1285):
    GIoU = I/U + U/M - 1, DIoU = I/U - |c1 - c2|^2 / D^2, with I/U the pinned rotated IoU (geometric truth), M the area of the convex hull of
    the eight vertices (dgal::merge :1021-1122 builds the same polygon with rotating calipers; here Andrew's monotone chain) and D their
    largest distance (dgal::dimension :941-982).  Small inputs only (Python loops).  PINNED to the reference's own giou2dr_forward /
    diou2dr_forward through tests/golden/iou_grad.npz (1e-12)."""
    b1, b2 = np.asarray(boxes1, np.float64), np.asarray(boxes2, np.float64)
    iou = iou2dr_truth(b1, b2)
    out = np.empty((len(b1), len(b2)))
    def verts(b):
        x, y, w, h, r = b
        c, s = np.cos(r), np.sin(r)
        return np.array([[x - w * c / 2 + h * s / 2, y - w * s / 2 - h * c / 2], [x + w * c / 2 + h * s / 2, y + w * s / 2 - h * c / 2],
                         [x + w * c / 2 - h * s / 2, y + w * s / 2 + h * c / 2], [x - w * c / 2 - h * s / 2, y - w * s / 2 + h * c / 2]])
    v1, v2 = [verts(b) for b in b1], [verts(b) for b in b2]
    for i in range(len(b1)):
        for j in range(len(b2)):
            m_area, diam = _hull_area_and_diameter(np.concatenate([v1[i], v2[j]]))
            a1, a2 = b1[i, 2] * b1[i, 3], b2[j, 2] * b2[j, 3]
            inter = iou[i, j] * (a1 + a2) / (1 + iou[i, j])
            u = a1 + a2 - inter
            if method == "grbox":
                out[i, j] = inter / u + u / m_area - 1
            else:
                out[i, j] = inter / u - ((b1[i, 0] - b2[j, 0]) ** 2 + (b1[i, 1] - b2[j, 1]) ** 2) / diam ** 2
    return out


def _ex_row(a, b, method):
    """values of `method` of one box a [1, 5] against b [M, 5], float64"""
    if method == "box":
        return iou2d(a, b)[0]
    if method == "rbox":
        return iou2dr_truth(a, b)[0]
    return iou2dr_ex(a, b, method)[0]


def iou_ex_local(boxes1, boxes2, method):
    """[N, M] values of box2d_iou's `method` ("box", "rbox", "grbox", "drbox") with each pair moved, in float64, into the frame of
    its first box's centre: the pinned forwards above (iou2d, iou2dr_truth, iou2dr_ex) without the cancellation of coordinates far
    from the origin.  Float32 boxes are widened exactly, so the shift is exact too.  One vectorised call per row."""
    b1, b2 = np.asarray(boxes1, np.float64), np.asarray(boxes2, np.float64)
    out = np.empty((len(b1), len(b2)))
    for i in range(len(b1)):
        a, b = b1[i:i + 1].copy(), b2.copy()
        b[:, :2] -= a[0, :2]
        a[0, :2] = 0
        out[i] = _ex_row(a, b, method)
    return out


def iou_ex_grad_local(boxes1, boxes2, method, h=1e-4, smooth_tol=1e-9):
    """Per-pair derivatives of iou_ex_local by five-point differences in each of the 5 box fields, taken in the local frame:
    returns (value [N, M], d1 [N, M, 5] = d value / d boxes1[i], d2 [N, M, 5] = d value / d boxes2[j], smooth bool [N, M]).
    A pair is smooth when the stencils at h and h/2 agree to `smooth_tol` in all ten derivatives; elsewhere (touching edges, a
    corner on an edge, a switch of hull edge or diameter, AABB min/max ties) the value has a kink within the stencil and no
    derivative to compare with.  Perturbing all of boxes2 at once is exact: value[i, j] depends on boxes2[j] alone."""
    b1, b2 = np.asarray(boxes1, np.float64), np.asarray(boxes2, np.float64)
    n, m = len(b1), len(b2)
    val, d1, d2, smooth = np.empty((n, m)), np.empty((n, m, 5)), np.empty((n, m, 5)), np.ones((n, m), bool)
    for i in range(n):
        a, b = b1[i:i + 1].copy(), b2.copy()
        b[:, :2] -= a[0, :2]
        a[0, :2] = 0
        val[i] = _ex_row(a, b, method)
        for side, d in ((0, d1), (1, d2)):
            for k in range(5):
                est = []
                for hh in (h, h / 2):
                    f = []
                    for s in (-2, -1, 1, 2):
                        a_, b_ = a.copy(), b.copy()
                        (b_ if side else a_)[:, k] += s * hh
                        f.append(_ex_row(a_, b_, method))
                    est.append((f[0] - 8 * f[1] + 8 * f[2] - f[3]) / (12 * hh))
                d[i, :, k] = est[0]
                smooth[i] &= np.abs(est[0] - est[1]) <= smooth_tol
    return val, d1, d2, smooth


def match_greedy(distance, src_scores, src_tags, dst_tags, thresholds):
    """ScoreMatcher.match (d3d/tracking/matcher.pyx:138-162) over BaseMatcher.match_by_order (:93-122) for one threshold set
    `thresholds[category]`: returns (src_assignment i32[N], dst_assignment i32[M]), -1 = unmatched.  The source order is
    np.flip(np.argsort(scores)) as in :143; the destination order of a source is ascending distance with ties to the lower index
    (the reference's unstable np.argsort leaves ties unspecified).  PARITY: restated, unpinned -- the matcher is a Cython module
    that needs the reference's whole object model and cannot be built here."""
    d = np.asarray(distance, np.float32)
    n, m = d.shape
    src_order = np.flip(np.argsort(np.asarray(src_scores, np.float64), kind="stable"))
    sa, da = np.full(n, -1, np.int32), np.full(m, -1, np.int32)
    for i in src_order:
        for j in np.argsort(d[i], kind="stable"):          # :145, :152-156
            if sa[i] >= 0:                                  # :104-105
                break
            if da[j] >= 0 or src_tags[i] != dst_tags[j]:    # :106-113
                continue
            if d[i, j] <= thresholds[dst_tags[j]]:          # :116-118
                sa[i], da[j] = j, i
    return sa, da


def nms2d(boxes, scores, iou_type=IOU_BOX, sup_type=SUP_HARD, iou_threshold=0.0, score_threshold=0.0,
          sup_param=0.0, alg=ALG_RC, cuda_score_rule=False, return_evals=False):
    """Suppressed mask u8[n]: d3d/box/nms.cpp:98-119 (order = stable descending argsort)."""
    dt = np.float32 if boxes.dtype == np.float32 else np.float64
    boxes = _boxes(boxes, dt)
    sc = np.ascontiguousarray(scores, dtype=dt).copy()
    order = np.argsort(-sc, kind="stable").astype(np.int64)
    sup = np.zeros(len(boxes), np.uint8)
    f = lib().orc_nms2d_f if dt == np.float32 else lib().orc_nms2d_d
    ev = f(_p(boxes), _p(sc), _p(order), C.c_int64(len(boxes)), C.c_int(iou_type), C.c_int(sup_type),
           C.c_float(iou_threshold), C.c_float(score_threshold), C.c_float(sup_param), C.c_int(alg),
           C.c_int(1 if cuda_score_rule else 0), _p(sup))
    return (sup.astype(bool), ev) if return_evals else sup.astype(bool)


def box2d_nms(boxes, scores, iou_method="box", supression_method="hard", iou_threshold=0, score_threshold=0,
              supression_param=0, precise=True, alg=ALG_RC, cuda_score_rule=False):
    """Front door: d3d/box/__init__.py:226-276; returns the KEEP mask bool[n]."""
    if precise:
        boxes, scores = boxes.astype(np.float64), scores.astype(np.float64)
    if scores.ndim == 2:
        scores = scores.max(axis=1)
    if boxes.size == 0:
        return np.zeros(0, bool)
    it = {"box": IOU_BOX, "rbox": IOU_RBOX}[iou_method]
    st = {"hard": SUP_HARD, "linear": SUP_LINEAR, "gaussian": SUP_GAUSSIAN}[supression_method]
    return ~nms2d(boxes, scores, it, st, iou_threshold, score_threshold, supression_param, alg, cuda_score_rule)


# ------------------------------------------------------------------ voxelization
def voxelize_dense(points, shape, bounds, max_points, max_voxels, reduction=0):
    """d3d/voxel/voxelize.cpp:45-199. Returns dict like the reference (pmask False where unset)."""
    pts = np.ascontiguousarray(points, np.float32)
    n, c = pts.shape
    shape = np.ascontiguousarray(shape, np.int32)
    bounds = np.ascontiguousarray(bounds, np.float32)
    voxels = np.zeros((max_voxels, max_points, c), np.float32)
    coords = np.zeros((max_voxels, 3), np.int64)
    pmask = np.zeros((max_voxels, max_points), np.uint8)
    npts = np.zeros(max_voxels, np.int32)
    agg = np.zeros((max_voxels, c), np.float32) if reduction else None
    nv = lib().orc_voxelize_dense(_p(pts), C.c_int64(n), C.c_int64(c), _p(shape), _p(bounds), C.c_int32(max_points),
                                  C.c_int32(max_voxels), C.c_int(reduction), _p(voxels), _p(coords), _p(pmask),
                                  _p(npts), _p(agg) if agg is not None else None)
    ret = dict(voxels=voxels[:nv], coords=coords[:nv], voxel_pmask=pmask[:nv].astype(bool), voxel_npoints=npts[:nv])
    if reduction:
        ret["aggregates"] = agg[:nv]
    return ret


def voxelize_sparse(points, voxel_size):
    """d3d/voxel/voxelize.cpp:288-335."""
    pts = np.ascontiguousarray(points, np.float32)
    n, c = pts.shape
    vs = np.ascontiguousarray(voxel_size, np.float32)
    mapping = np.empty(n, np.int64)
    coords = np.empty((max(n, 1), 3), np.int64)
    npts = np.empty(max(n, 1), np.int32)
    nv = lib().orc_voxelize_sparse(_p(pts), C.c_int64(n), C.c_int64(c), _p(vs), _p(mapping), _p(coords), _p(npts))
    return dict(points_mapping=mapping, coords=coords[:nv].copy(), voxel_npoints=npts[:nv].copy())


def voxelize_filter(points, mapping, coords, npoints, coords_bound, min_points, max_points, max_voxels,
                    pfilter, vfilter):
    """d3d/voxel/voxelize.cpp:337-484."""
    pts = np.ascontiguousarray(points, np.float32)
    n = len(pts)
    nv = len(coords)
    mapping = np.ascontiguousarray(mapping, np.int64)
    coords = np.ascontiguousarray(coords, np.int64)
    npoints = np.ascontiguousarray(npoints, np.int32)
    bnd = None if coords_bound is None else np.ascontiguousarray(coords_bound, np.int64)
    out_mask = np.empty(max(n, 1), np.int64)
    out_map = np.empty(max(n, 1), np.int64)
    out_np = np.empty(max(nv, 1), np.int32)
    out_co = np.empty((max(nv, 1), 3), np.int64)
    k = C.c_int64(0)
    v = lib().orc_voxelize_filter(C.c_int64(n), _p(mapping), _p(coords), _p(npoints), C.c_int64(nv),
                                  _p(bnd) if bnd is not None else None, C.c_int32(min_points), C.c_int32(max_points),
                                  C.c_int32(max_voxels), C.c_int(pfilter), C.c_int(vfilter), _p(out_mask), _p(out_map),
                                  _p(out_np), _p(out_co), C.byref(k))
    k = k.value
    return dict(points=pts[out_mask[:k]], points_mask=out_mask[:k].copy(), points_mapping=out_map[:k].copy(),
                voxel_npoints=out_np[:v].copy(), coords=out_co[:v].copy())


_RED = {None: 0, "none": 0, "mean": 1, "max": 2, "min": 3}
_PF = {None: 0, "none": 0, "trim": 1}
_VF = {None: 0, "none": 0, "trim": 1, "descending": 2}


class VoxelGenerator:
    """d3d/voxel/__init__.py:12-104 restated on numpy + the C oracle (fp32 derivations kept identical)."""

    def __init__(self, bounds, shape, min_points=0, max_points=30, max_voxels=20000, max_points_filter=None,
                 max_voxels_filter=None, reduction=None, dense=False):
        self.bounds = np.asarray(bounds, np.float32)
        self.shape = np.asarray(shape, np.int32)
        ba = self.bounds.reshape(3, 2)
        self.size = ((ba[:, 1] - ba[:, 0]) / self.shape.astype(np.float32)).astype(np.float32)
        dist = (ba[:, 0] / self.size).astype(np.float32)
        if np.any(np.abs(np.round(dist) - dist) > 1e-3):
            raise ValueError("The voxelization grids is not aligned with the origin")
        self.offset = np.round(dist).astype(np.int32)
        self.vbounds = np.round((ba / self.size.reshape(3, 1)).astype(np.float32)).astype(np.int64)
        self.min_points, self.max_points, self.max_voxels = min_points, max_points, max_voxels
        self.pf = _PF[max_points_filter.lower() if max_points_filter else None]
        self.vf = _VF[max_voxels_filter.lower() if max_voxels_filter else None]
        self.red = _RED[reduction.lower() if reduction else None]
        self.dense = dense

    def __call__(self, points):
        if self.dense:
            return voxelize_dense(points, self.shape, self.bounds, self.max_points, self.max_voxels, self.red)
        sp = voxelize_sparse(points, self.size)
        ret = voxelize_filter(points, sp["points_mapping"], sp["coords"], sp["voxel_npoints"], self.vbounds,
                              self.min_points, self.max_points, self.max_voxels, self.pf, self.vf)
        ret["coords"] = ret["coords"] - self.offset.astype(np.int64)
        return ret


# ------------------------------------------------------------------ aligned scatter
def scatter_forward(coord, image, atype):
    """d3d/point/scatter.cpp:79-134,175-188. atype: 1 MEAN, 2 LINEAR."""
    dt = np.float32 if image.dtype == np.float32 else np.float64
    coord = np.ascontiguousarray(coord, dt)
    image = np.ascontiguousarray(image, dt)
    n, dim = coord.shape[0], coord.shape[1] - 1
    dims = np.asarray(image.shape[2:], np.int64)
    out = np.empty((n, image.shape[1]), dt)
    f = lib().orc_scatter_fwd_f32 if dt == np.float32 else lib().orc_scatter_fwd_f64
    f(_p(coord), C.c_int64(n), C.c_int(dim), _p(image), C.c_int64(image.shape[0]), C.c_int64(image.shape[1]),
      _p(dims), C.c_int(atype), _p(out))
    return out


def scatter_backward(coord, grad, atype, image_shape):
    """d3d/point/scatter.cpp:136-172,190-201 (image_grad starts at zero, d3d/point/__init__.py:32)."""
    dt = np.float32 if grad.dtype == np.float32 else np.float64
    coord = np.ascontiguousarray(coord, dt)
    grad = np.ascontiguousarray(grad, dt)
    n, dim = coord.shape[0], coord.shape[1] - 1
    dims = np.asarray(image_shape[2:], np.int64)
    ig = np.zeros(image_shape, dt)
    f = lib().orc_scatter_bwd_f32 if dt == np.float32 else lib().orc_scatter_bwd_f64
    f(_p(coord), C.c_int64(n), C.c_int(dim), _p(grad), C.c_int64(image_shape[0]), C.c_int64(image_shape[1]),
      _p(dims), C.c_int(atype), _p(ig))
    return ig
