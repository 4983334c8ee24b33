"""Inputs and reference sums shared by the CPU (host twin) and GPU checks of the differentiable IoU family: boxes moved far from
the origin, near-collinear corners, equivalent parametrisations of a box, and the gradient sums of the local-frame float64
reference (oracle.iou_ex_grad_local)."""
import numpy as np

METHODS = ("box", "rbox", "grbox", "drbox")
OFFSETS = {np.float32: (0.0, 75.0, 1e3), np.float64: (0.0, 75.0, 1e3, 1e5)}
# values | gradients relative to max(1, max |ref|)
TOL = {np.float32: (1e-5, 1e-4), np.float64: (1e-10, 1e-8)}

# fp32 pair whose corners A1, A2, B2 are nearly collinear: a hull built from per-pair tolerances took both (A1, B2) and (A2, B2) as edges
# and returned GIoU 0.234899 for 0.241330
PINNED_A = np.array([[-1.11077880859375, 4.67926025390625, 1.8252308368682861, 1.940333604812622, 3.51875901222229]], np.float32)
PINNED_B = np.array([[0.12176513671875, 4.45025634765625, 3.4699227809906006, 2.6391003131866455, 3.306314468383789]], np.float32)

EPS = (-1e-3, -1e-5, -1e-7, -1e-9, 0.0, 1e-9, 1e-7, 1e-5, 1e-3)
TURNS = (-1e-3, -1e-5, -1e-7, 1e-7, 1e-5, 1e-3)


def shifted(a, b, off, rng):
    """both sides moved by `off` metres in a random direction (the geometry of every pair is unchanged)"""
    th = rng.random() * 2 * np.pi
    d = np.array([off * np.cos(th), off * np.sin(th), 0, 0, 0])
    return a + d, b + d


def collinear_family(rng, slides=(-0.9, -0.3, 0.0, 0.45, 1.2)):
    """A [1, 5] and B [len(EPS) * 2 * len(slides), 5]: B has A's heading and one edge on the line of one of A's edges, offset along the
    normal by eps * (A's height) and slid along the edge.  'outer' puts B's bottom edge on A's top edge line (B beside A, touching at
    eps = 0), 'inner' puts B's top edge on A's top edge line (B overlapping A, flush).  Column index = (slide, kind, eps) row-major."""
    w, h, r = 2.0 + 2 * rng.random(), 1.0 + rng.random(), (rng.random() - .5) * 6
    wb, hb = 1.0 + 2 * rng.random(), 0.5 + rng.random()
    u, v = np.array([np.cos(r), np.sin(r)]), np.array([-np.sin(r), np.cos(r)])
    rows = []
    for t in slides:
        for kind in (1, -1):
            for e in EPS:
                c = (h / 2 + kind * hb / 2 + e * h) * v + t * w * u
                rows.append([c[0], c[1], wb, hb, r])
    return np.array([[0, 0, w, h, r]]), np.array(rows)


def turned_family(rng):
    """A [1, 5] and B [len(TURNS), 5]: B's corner 0 on A's corner 1 and B turned by delta from A's heading about that corner, so
    that A0, A1 = B0, B1 and A2, B3 are nearly collinear"""
    w, h, r = 2.0 + 2 * rng.random(), 1.0 + rng.random(), (rng.random() - .5) * 6
    wb, hb = 1.0 + 2 * rng.random(), 0.5 + 2 * rng.random()
    a1 = np.array([w / 2 * np.cos(r) + h / 2 * np.sin(r), w / 2 * np.sin(r) - h / 2 * np.cos(r)])
    rows = []
    for d in TURNS:
        q = r + d
        c = a1 + wb / 2 * np.array([np.cos(q), np.sin(q)]) + hb / 2 * np.array([-np.sin(q), np.cos(q)])
        rows.append([c[0], c[1], wb, hb, q])
    return np.array([[0, 0, w, h, r]]), np.array(rows)


def equivalents(b):
    """the same rectangles written three other ways: turned by pi, by 2 pi, and with w, h swapped and turned by pi / 2"""
    p, q, s = b.copy(), b.copy(), b.copy()
    p[:, 4] += np.pi
    q[:, 4] += 2 * np.pi
    s[:, 2], s[:, 3] = b[:, 3], b[:, 2]
    s[:, 4] += np.pi / 2
    return p, q, s


def reference(oracle, a, b, method, up):
    """(value [N, M], grad1 [N, 5], grad2 [M, 5], upstream gradient with the non-smooth pairs zeroed, smooth mask) of the local-frame
    float64 reference on the float64 widening of a, b and up"""
    v, d1, d2, smooth = oracle.iou_ex_grad_local(a.astype(np.float64), b.astype(np.float64), method)
    upm = np.where(smooth, up, 0).astype(up.dtype)
    u = upm.astype(np.float64)
    return v, np.einsum("ij,ijk->ik", u, d1), np.einsum("ij,ijk->jk", u, d2), upm, smooth


def rel_err(got, ref):
    return float(np.abs(np.asarray(got, np.float64) - ref).max() / max(1.0, np.abs(ref).max())) if ref.size else 0.0
