"""Inputs and reference sums shared by the CPU (host twin) and GPU checks of the signed point-to-box distance (box2dr_pdist, dist.cuh):
boxes and points moved far from the origin, points on the lines through edges, exact ties, special headings, equivalent
parametrisations, zero-size boxes, a lidar-scale scene, and the gradient sums of the local-frame float64 reference
(oracle.pdist2dr_grad_local)."""
import numpy as np

from conftest import gen_boxes

OFFSETS = {np.float32: (0.0, 75.0, 1e3), np.float64: (0.0, 75.0, 1e3, 1e5)}
# values | gradients, both relative to max(1, |ref|): per pair for values (a distance of 150 m in fp32 carries ulps of 1.5e-5), over
# the whole array for gradient sums
TOL = {np.float32: (1e-5, 1e-4), np.float64: (1e-10, 1e-8)}
STEPS = (1e-9, 1e-7, 1e-5, 1e-3, 1e-1, 1.0)
HEADINGS = (0.0, np.pi / 2, -np.pi / 2, np.pi, 3 * np.pi / 2, 2 * np.pi, 1e-9, -1e-9, 1e-17, -1e-17)
ORDER = (3, 0, 1, 2)   # edge loop order: equal distances go to the first of these

# Pairs where the reference's pdist2dr (dgal's distance(Poly2, Point2)) is wrong, with the truth: a point on the line through an edge,
# outside the box, comes out positive (the adjacent edges tie and the first one's line gives the sign), and at a heading of pi / 2 the
# projection divides by cos(pi / 2) = 6e-17
REF_WRONG = [  # (point, box, reference's value, truth)
    ((3.0, -1.0), (0, 0, 4, 2, 0), 1.0, -1.0),
    ((2.0, 2.0), (0, 0, 4, 2, 0), 1.0, -1.0),
    ((-2.0, 2.5), (0, 0, 4, 2, 0), 1.5, -1.5),
]


def val_err(got, ref):
    """largest |got - ref| / max(1, |ref|) over the pairs"""
    ref = np.asarray(ref, np.float64)
    return float((np.abs(np.asarray(got, np.float64) - ref) / np.maximum(1.0, np.abs(ref))).max()) if ref.size else 0.0


def rel_err(got, ref):
    return float(np.abs(np.asarray(got, np.float64) - ref).max() / max(1.0, np.abs(ref).max())) if ref.size else 0.0


def near_points(rng, boxes, n):
    """n points scattered over the boxes' surroundings: each near a random box, up to 1.5 half diagonals from its centre"""
    k = rng.integers(0, len(boxes), n)
    rad = 0.75 * np.hypot(boxes[k, 2], boxes[k, 3]) + 0.5
    return boxes[k, :2] + (rng.random((n, 2)) * 2 - 1) * rad[:, None]


def shifted(points, boxes, off, rng):
    """points and boxes moved by `off` metres in a random direction (every pair's geometry is unchanged)"""
    th = rng.random() * 2 * np.pi
    d = np.array([off * np.cos(th), off * np.sin(th)])
    b = boxes.copy()
    b[:, :2] += d
    return points + d, b


def to_world(box, q):
    """local points q [K, 2] of box (x, y, w, h, r) in the caller's frame"""
    c, s = np.cos(box[4]), np.sin(box[4])
    return np.stack([box[0] + c * q[:, 0] - s * q[:, 1], box[1] + s * q[:, 0] + c * q[:, 1]], 1)


def edge_line_points(box):
    """local points (+-(hw + s), +-hh) and (+-hw, +-(hh + s)) for s in STEPS: outside the box on the line through an edge, at distance s
    from a corner.  Returns (points [8 * len(STEPS), 2] in the caller's frame, s per point)"""
    hw, hh = abs(box[2]) / 2, abs(box[3]) / 2
    q, d = [], []
    for sx in (-1, 1):
        for sy in (-1, 1):
            for s in STEPS:
                q += [(sx * (hw + s), sy * hh), (sx * hw, sy * (hh + s))]
                d += [s, s]
    return to_world(box, np.array(q)), np.array(d)


def tie_cases():
    """(boxes [M, 5], points [N, 2], expected edge [M, N]) with heading 0 and dyadic coordinates, so that every local offset is exact and
    ties are exact: the centre, the diagonals of squares, the corners, the edge midpoints and points on the lines through edges.  The
    expected edge is the first edge of ORDER among those whose distance is the box's distance."""
    boxes = np.array([[1.5, -2.25, 4, 4, 0], [1.5, -2.25, -4, 4, 0], [1.5, -2.25, 4, -4, 0], [1.5, -2.25, 4, 2, 0], [1.5, -2.25, -4, -2, 0]])
    local = [(0, 0)]
    for t in (0.5, 1.0, 1.75):
        local += [(t, t), (-t, t), (t, -t), (-t, -t)]
    for hx in (-1, 0, 1):
        for hy in (-1, 0, 1):
            local.append((hx, hy))                                   # unit offsets: scaled per box below
    pts, edges = [], []
    for b in boxes:
        hw, hh = abs(b[2]) / 2, abs(b[3]) / 2
        q = [p for p in local[:13] if abs(p[0]) <= hw and abs(p[1]) <= hh]
        q += [(hx * hw, hy * hh) for hx, hy in local[13:]]           # centre, edge midpoints, corners
        q += [(hw + .5, hh), (-hw, -hh - .25), (hw + .5, 0), (0, -hh - 1)]
        pts.append([(b[0] + x, b[1] + y) for x, y in q])
        edges.append([_expected_edge(b, x, y) for x, y in q])
    allp = np.concatenate([np.array(p) for p in pts])
    exp = np.full((len(boxes), len(allp)), 255, np.uint8)   # only the points made for a box are checked against it
    o = 0
    for i, e in enumerate(edges):
        exp[i, o:o + len(e)] = e
        o += len(e)
    return boxes, allp, exp


def _expected_edge(b, x, y):
    """edge by exact enumeration of the four segment distances of the axis-aligned box b at the local point (x, y)"""
    w, h = b[2], b[3]
    v = [(-w / 2, -h / 2), (w / 2, -h / 2), (w / 2, h / 2), (-w / 2, h / 2)]
    dist = []
    for k in range(4):
        (ax, ay), (bx, by) = v[k], v[(k + 1) % 4]
        if ax == bx:   # vertical edge
            dist.append(np.hypot(x - ax, max(min(ay, by) - y, 0, y - max(ay, by))))
        else:
            dist.append(np.hypot(y - ay, max(min(ax, bx) - x, 0, x - max(ax, bx))))
    dmin = min(dist)
    return next(k for k in ORDER if dist[k] == dmin)


def heading_cases(rng):
    """boxes with the headings of HEADINGS, centred at the origin, on either axis and off them, and points around them"""
    rows = []
    for r in HEADINGS:
        for cx, cy in ((0, 0), (7, 0), (0, -7), (3.25, -5.5)):
            rows.append([cx, cy, 4, 2, r])
    b = np.array(rows)
    return near_points(rng, b, 600), b


def zero_boxes():
    """boxes with w = 0, h = 0 and both: a segment (minus the distance to it) and a point (minus the distance to the centre)"""
    return np.array([[0.5, -1, 0, 3, 0.4], [0.5, -1, 2, 0, -1.1], [0.5, -1, 0, 0, 0.7], [0.5, -1, 0, 3, 0], [0.5, -1, 0, 0, 0]])


def equivalents(b):
    """the same rectangles written five other ways: turned by pi, by 2 pi, w and h swapped and turned by pi / 2, w negated, h negated"""
    p, q, s, u, v = b.copy(), b.copy(), b.copy(), b.copy(), b.copy()
    p[:, 4] += np.pi
    q[:, 4] += 2 * np.pi
    s[:, 2], s[:, 3] = b[:, 3], b[:, 2]
    s[:, 4] += np.pi / 2
    u[:, 2] *= -1
    v[:, 3] *= -1
    return p, q, s, u, v


def lidar_scene():
    """the benchmark's lidar cloud (20 000 points within 80 m, bench.lidar) against 200 car-sized proposals (bench.proposals), float32"""
    import bench
    pts = np.ascontiguousarray(bench.lidar(3, 20000)[:, :2])
    boxes = bench.proposals(4, 200, 50)[0].astype(np.float32)
    return pts, boxes


def reference(oracle, points, boxes, up):
    """(value [M, N], grad_points [N, 2], grad_boxes [M, 5], upstream gradient with the non-smooth pairs zeroed, smooth mask) of the
    local-frame float64 reference on the float64 widening of points, boxes and up"""
    v, dp, db, smooth = oracle.pdist2dr_grad_local(points.astype(np.float64), boxes.astype(np.float64))
    upm = np.where(smooth, up, 0).astype(up.dtype)
    u = upm.astype(np.float64)
    return v, np.einsum("ij,ijk->jk", u, dp), np.einsum("ij,ijk->ik", u, db), upm, smooth


def translation_case(off, dt):
    """40 points x 12 boxes near the origin, moved by `off` in a random direction, in dtype dt, with an upstream gradient"""
    rng = np.random.default_rng(int(off) + 3)
    b = gen_boxes(rng, 12) + [0, 0, .2, .2, 0]
    p, b = shifted(near_points(rng, b, 40), b, off, rng)
    return p.astype(dt), b.astype(dt), rng.normal(size=(12, 40)).astype(dt)


# ------------------------------------------------------------------ checks shared by the host twin and the GPU
# `run(points, boxes, up)` returns (value [M, N], edge index [M, N], gradient of sum(up * value) in the points [N, 2] and boxes [M, 5]),
# in the dtype of its inputs.

def check_translation(run, oracle, dt):
    """the same 40 x 12 pairs at growing distance from the origin: values, both gradients and the edge index"""
    vt, gt = TOL[dt]
    worst = {}
    for off in OFFSETS[dt]:
        p, b, up = translation_case(off, dt)
        v, gp, gb, upm, smooth = reference(oracle, p, b, up)
        assert smooth.mean() > 0.9, off
        kv, ke, kp, kb = run(p, b, upm)
        e = (val_err(kv, v), rel_err(kp, gp), rel_err(kb, gb))
        worst[off] = e
        assert e[0] <= vt and e[1] <= gt and e[2] <= gt, (off, e)
        ref_e = oracle.pdist2dr_local(p, b, return_iedge=True)[1]
        assert np.array_equal(ke[smooth], ref_e[smooth]), off
    return worst


def check_edge_lines(run, oracle, dt):
    """points outside the box on the lines through its edges, s = 1e-9 .. 1 from a corner, on turned and shifted boxes: values equal
    the reference and are negative (the reference's pdist2dr makes them positive); in fp64 they are -s, so continuous in s"""
    vt = TOL[dt][0]
    rng = np.random.default_rng(41)
    for off in OFFSETS[dt]:
        for box in ([0, 0, 4, 2, 0], [0, 0, 4, 2, np.pi / 2], [2, -1, 3, 1.5, 0.3], [0, 0, 2, 2, -2.2], [5, 5, -4, 2, 1.0]):
            b = np.array([box], np.float64)
            p, s = edge_line_points(b[0])
            p, b = shifted(p, b, off, rng)
            p, b = p.astype(dt), b.astype(dt)
            kv = run(p, b, np.zeros((1, len(p)), dt))[0][0]
            ref = oracle.pdist2dr_local(p, b)[0]
            assert val_err(kv, ref) <= vt, (off, box, val_err(kv, ref))
            if dt == np.float64:
                assert np.abs(kv + s).max() <= vt * max(1.0, off * 1e-4) and (kv < 0).all(), (off, box)
            else:
                assert (kv[s >= 1e-3] < 0).all(), (off, box)


def check_ties(run, oracle):
    """exact ties at heading 0 (centre of a square, diagonals, corners, edge midpoints, lines through edges; negative w and h): the
    edge index is the first of the loop order 3, 0, 1, 2 among the edges that realise the distance, and so is the reference's"""
    b, p, exp = tie_cases()
    sel = exp != 255
    ref_v, ref_e = oracle.pdist2dr_local(p, b, return_iedge=True)
    assert np.array_equal(ref_e[sel], exp[sel])
    for dt in (np.float64, np.float32):
        kv, ke, _, _ = run(p.astype(dt), b.astype(dt), np.zeros(exp.shape, dt))
        assert np.array_equal(ke[sel], exp[sel]), dt
        assert np.array_equal(kv[sel], ref_v[sel]), dt   # dyadic inputs: every operation is exact
    assert exp[0, 0] == 3   # the centre of a square: all four edges tie


def check_headings(run, oracle, dt):
    """headings 0, +-pi/2, pi, 3 pi/2, 2 pi, +-1e-9, +-1e-17 on boxes centred at the origin, on either axis and off them"""
    vt, gt = TOL[dt]
    p, b = heading_cases(np.random.default_rng(43))
    p, b = p.astype(dt), b.astype(dt)
    up = np.random.default_rng(44).normal(size=(len(b), len(p))).astype(dt)
    v, gp, gb, upm, smooth = reference(oracle, p, b, up)
    assert smooth.mean() > 0.9
    kv, _, kp, kb = run(p, b, upm)
    e = (val_err(kv, v), rel_err(kp, gp), rel_err(kb, gb))
    assert e[0] <= vt and e[1] <= gt and e[2] <= gt, e


def check_equivalent_boxes(run):
    """(x, y, w, h, r + pi), (x, y, w, h, r + 2 pi), (x, y, h, w, r + pi / 2), (x, y, -w, h, r), (x, y, w, -h, r) are the same rectangle:
    the same values and point gradients to 1e-12 in fp64"""
    rng = np.random.default_rng(45)
    b = gen_boxes(rng, 10) + [0, 0, .3, .3, 0]
    p = near_points(rng, b, 200)
    up = rng.normal(size=(10, 200))
    v, _, gp, _ = run(p, b, up)
    for i, e in enumerate(equivalents(b)):
        ve, _, gpe, _ = run(p, e, up)
        assert np.abs(ve - v).max() <= 1e-12 and rel_err(gpe, gp) <= 1e-12, i


def check_zero_size(run, oracle, dt):
    """w = 0: minus the distance to the segment; w = h = 0: -|p - c|.  Values against the reference; gradients where smooth"""
    vt, gt = TOL[dt]
    rng = np.random.default_rng(47)
    b = zero_boxes()
    p = np.concatenate([b[:, :2] + (rng.random((len(b), 2)) - .5) * 6, near_points(rng, b + [0, 0, 1, 1, 0], 100)]).astype(dt)
    b = b.astype(dt)
    up = rng.normal(size=(len(b), len(p))).astype(dt)
    v, gp, gb, upm, smooth = reference(oracle, p, b, up)
    assert (v[2:3] <= 0).all() and (v[4:5] <= 0).all()
    c = b[2, :2].astype(np.float64)
    assert np.abs(v[2] + np.hypot(p[:, 0] - c[0], p[:, 1] - c[1])).max() <= 1e-12
    kv, _, kp, kb = run(p, b, upm)
    e = (val_err(kv, v), rel_err(kp, gp), rel_err(kb[:, [0, 1, 4]], gb[:, [0, 1, 4]]))
    assert e[0] <= vt and e[1] <= gt and e[2] <= gt, e


def check_lidar_scene(run, oracle):
    """20 000 lidar points x 200 proposals in fp32, all 4 M pairs against the reference; gradients on the first 2 000 points"""
    vt, gt = TOL[np.float32]
    p, b = lidar_scene()
    kv, ke, _, _ = run(p, b, np.zeros((len(b), len(p)), np.float32))
    ref = oracle.pdist2dr_local(p, b)
    assert val_err(kv, ref) <= vt, val_err(kv, ref)
    ps = p[:2000]
    up = np.random.default_rng(49).normal(size=(len(b), len(ps))).astype(np.float32)
    v, gp, gb, upm, smooth = reference(oracle, ps, b, up)
    _, _, kp, kb = run(ps, b, upm)
    assert rel_err(kp, gp) <= gt and rel_err(kb, gb) <= gt, (rel_err(kp, gp), rel_err(kb, gb))
