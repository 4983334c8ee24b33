"""CPU check of the pair math of the signed point-to-box distance: d3d_b200/csrc/dist.cuh compiled as host code (tests/host_twin)
against the local-frame float64 reference (oracle.pdist2dr_local / pdist2dr_grad_local).  Values, edge indices and both gradients, far
from the origin, on the lines through edges, at exact ties and special headings, on equivalent and zero-size boxes and on a lidar-scale
scene.  The GPU tests (test_pdist_parity.py) run the same checks on the kernels.  Also pins where the reference's own pdist2dr (dgal's
distance(Poly2, Point2)) departs from the truth: the deviation P1 of SURVEY.md 8(c)."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import pdist_cases as P
from conftest import golden

HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def twin():
    subprocess.check_call(["make", "-s", "-C", os.path.join(HERE, "host_twin")])
    lib = C.CDLL(os.path.join(HERE, "host_twin", "libtwin.so"))

    def run(points, boxes, up):
        """(values [M, N], edge [M, N], grad points [N, 2], grad boxes [M, 5]) as pdist_fwd_kernel / pdist_bwd_kernel compute them"""
        p, b = np.ascontiguousarray(points), np.ascontiguousarray(boxes)
        dt = p.dtype
        n, m = len(p), len(b)
        up = np.ascontiguousarray(up, dt)
        out, e, gp, gb = np.empty((m, n), dt), np.empty((m, n), np.uint8), np.empty((n, 2), dt), np.empty((m, 5), dt)
        f = lib.twin_pdist_f32 if dt == np.float32 else lib.twin_pdist_f64
        ptr = lambda x: x.ctypes.data_as(C.c_void_p)  # noqa: E731
        f(ptr(p), C.c_long(n), ptr(b), C.c_long(m), ptr(up), ptr(out), ptr(e), ptr(gp), ptr(gb))
        return out, e, gp, gb
    return run


DTS = pytest.mark.parametrize("dt", [np.float32, np.float64], ids=["f32", "f64"])


@DTS
def test_translation(twin, oracle, dt):
    P.check_translation(twin, oracle, dt)


@DTS
def test_edge_lines(twin, oracle, dt):
    P.check_edge_lines(twin, oracle, dt)


def test_ties(twin, oracle):
    P.check_ties(twin, oracle)


@DTS
def test_headings(twin, oracle, dt):
    P.check_headings(twin, oracle, dt)


def test_equivalent_boxes(twin):
    P.check_equivalent_boxes(twin)


@DTS
def test_zero_size(twin, oracle, dt):
    P.check_zero_size(twin, oracle, dt)


def test_lidar_scene(twin, oracle):
    P.check_lidar_scene(twin, oracle)


def test_reference_deviation_p1(oracle):
    """The reference's pdist2dr is not the signed distance (SURVEY.md 8(c), P1), and box2dr_pdist follows the truth instead:
    - points on the line through an edge, outside the box, come out positive (the pairs of REF_WRONG);
    - at a heading of pi / 2 a third of the points around a box centred at the origin are wrong, by metres, in fp64;
    - the committed fixture pdist.npz, written by the reference, holds such values."""
    for p, b, ref_v, truth in P.REF_WRONG:
        pts, box = np.array([p]), np.array([b], np.float64)
        assert oracle.pdist2dr(pts, box)[0, 0] == ref_v and oracle.pdist2dr_local(pts, box)[0, 0] == truth, (p, b)
    rng = np.random.default_rng(0)
    q, bb = (rng.random((2000, 2)) - .5) * 10, np.array([[0., 0, 4, 2, np.pi / 2]])
    err = np.abs(oracle.pdist2dr(q, bb) - oracle.pdist2dr_local(q, bb))
    assert (err > 1e-6).mean() > 0.3 and err.max() > 5
    g = golden("pdist.npz")
    for tag, tol, wrong in (("f32", 1e-4, 27), ("f64", 1e-9, 23)):
        err = np.abs(g[f"{tag}.dist"] - oracle.pdist2dr_local(g[f"{tag}.points"], g[f"{tag}.boxes"]))
        assert (err > tol).sum() == wrong and err.max() > 0.3, tag
