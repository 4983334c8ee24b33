"""CPU check of the pair math of the differentiable IoU family: d3d_b200/csrc/iou_grad.cuh compiled as host code (tests/host_twin)
against the local-frame float64 reference (oracle.iou_ex_local / iou_ex_grad_local).  Values and both gradients, for the four methods,
far from the origin, on near-collinear corners and on equivalent parametrisations of the same boxes.  The GPU tests
(test_iou_grad_parity.py) run the same checks on the kernels."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from conftest import gen_boxes
from iou_ex_cases import (METHODS, OFFSETS, TOL, PINNED_A, PINNED_B, EPS, shifted, collinear_family, turned_family, equivalents,
                          reference, rel_err)

HERE = os.path.dirname(os.path.abspath(__file__))
TYPE = {"box": 0, "rbox": 1, "grbox": 2, "drbox": 3}   # GT_BOX .. GT_DIOU of iou_grad.cuh


@pytest.fixture(scope="module")
def twin_ex():
    subprocess.check_call(["make", "-s", "-C", os.path.join(HERE, "host_twin")])
    lib = C.CDLL(os.path.join(HERE, "host_twin", "libtwin.so"))

    def run(b1, b2, method, up=None):
        """(values [N, M], grad1 [N, 5], grad2 [M, 5]) as iou_ex_fwd_kernel / iou_bwd_kernel compute them"""
        b1, b2 = np.ascontiguousarray(b1), np.ascontiguousarray(b2)
        dt = b1.dtype
        up = np.zeros((len(b1), len(b2)), dt) if up is None else np.ascontiguousarray(up, dt)
        out, g1, g2 = np.empty((len(b1), len(b2)), dt), np.empty((len(b1), 5), dt), np.empty((len(b2), 5), dt)
        f = lib.twin_iou_ex_f32 if dt == np.float32 else lib.twin_iou_ex_f64
        p = lambda x: x.ctypes.data_as(C.c_void_p)  # noqa: E731
        f(p(b1), C.c_long(len(b1)), p(b2), C.c_long(len(b2)), C.c_int(TYPE[method]), p(up), p(out), p(g1), p(g2))
        return out, g1, g2
    return run


@pytest.mark.parametrize("dt", [np.float32, np.float64], ids=["f32", "f64"])
def test_translation(twin_ex, oracle, dt):
    """the same 12 x 10 pairs at growing distance from the origin: the pair code works in a box's own frame, so nothing may move"""
    vt, gt = TOL[dt]
    for off in OFFSETS[dt]:
        rng = np.random.default_rng(int(off) + 7)
        a, b = shifted(gen_boxes(rng, 12), gen_boxes(rng, 10), off, rng)
        a, b = a.astype(dt), b.astype(dt)
        up = rng.normal(size=(12, 10)).astype(dt)
        for m in METHODS:
            v, g1, g2, upm, smooth = reference(oracle, a, b, m, up)
            assert smooth.mean() > 0.8, (m, off)
            tv, tg1, tg2 = twin_ex(a, b, m, upm)
            errs = (np.abs(tv - v).max(), rel_err(tg1, g1), rel_err(tg2, g2))
            assert errs[0] <= vt and errs[1] <= gt and errs[2] <= gt, (m, off, errs)


def test_pinned_near_collinear_pair(twin_ex, oracle):
    a, b = PINNED_A, PINNED_B
    for m in ("grbox", "drbox", "rbox"):
        ref = oracle.iou_ex_local(a.astype(np.float64), b.astype(np.float64), m)
        assert abs(twin_ex(a, b, m)[0][0, 0] - ref[0, 0]) <= 1e-5, m
        assert abs(twin_ex(a.astype(np.float64), b.astype(np.float64), m)[0][0, 0] - ref[0, 0]) <= 1e-10, m
    assert abs(oracle.iou_ex_local(a.astype(np.float64), b.astype(np.float64), "grbox")[0, 0] - 0.241330) < 1e-6


@pytest.mark.parametrize("dt", [np.float32, np.float64], ids=["f32", "f64"])
def test_near_collinear_families(twin_ex, oracle, dt):
    """B flush with or touching one of A's edges (offset eps along the normal, slid along the edge) and B turned by a tiny angle
    about a corner it shares with A: GIoU / DIoU / IoU values match the reference and move continuously with eps"""
    vt = TOL[dt][0]
    rng = np.random.default_rng(21)
    for off in (0.0, 75.0):
        for fam in range(3):
            for a, b in (collinear_family(rng), turned_family(rng)):
                a, b = shifted(a, b, off, rng)
                a, b = a.astype(dt), b.astype(dt)
                for m in ("rbox", "grbox", "drbox"):
                    ref = oracle.iou_ex_local(a, b, m)[0]
                    got, g1, g2 = twin_ex(a, b, m, np.ones((1, len(b)), dt))
                    assert np.abs(got[0] - ref).max() <= vt, (m, off, fam, np.abs(got[0] - ref).max())
                    assert np.isfinite(g1).all() and np.isfinite(g2).all()
                    if len(b) > len(EPS):   # the eps sweeps of collinear_family: steps of the value follow the reference's
                        st, sr = np.diff(got[0].reshape(-1, len(EPS)), axis=1), np.diff(ref.reshape(-1, len(EPS)), axis=1)
                        assert np.abs(st - sr).max() <= 2 * vt, (m, off, fam)


def test_equivalent_boxes(twin_ex):
    """(x, y, w, h, r + pi), (x, y, w, h, r + 2 pi) and (x, y, h, w, r + pi / 2) are the same rectangle: same values and the same
    gradient in x and y, on either side"""
    rng = np.random.default_rng(5)
    a, b = gen_boxes(rng, 12) + [0, 0, .3, .3, 0], gen_boxes(rng, 10) + [0, 0, .3, .3, 0]
    up = rng.normal(size=(12, 10))
    for m in ("rbox", "grbox", "drbox"):
        v, g1, g2 = twin_ex(a, b, m, up)
        for e in equivalents(b):
            ve, g1e, g2e = twin_ex(a, e, m, up)
            assert np.abs(ve - v).max() <= 1e-12 and rel_err(g1e, g1) <= 1e-12 and rel_err(g2e[:, :2], g2[:, :2]) <= 1e-12, m
        for e in equivalents(a):
            ve, g1e, g2e = twin_ex(e, b, m, up)
            assert np.abs(ve - v).max() <= 1e-12 and rel_err(g1e[:, :2], g1[:, :2]) <= 1e-12 and rel_err(g2e, g2) <= 1e-12, m
