import hashlib
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def golden(name):
    return np.load(os.path.join(GOLDEN, name), allow_pickle=False)


@pytest.fixture(scope="session")
def oracle():
    """The CPU oracle (checker).  Built on demand with gcc."""
    from oracle import oracle as O
    O.lib()
    return O


def gen_boxes(rng, n, spread=10.0):
    """Reference benchmark distribution (test/compare/benchmark_riou.py:70-74)."""
    return np.stack([(rng.random(n) - .5) * spread, (rng.random(n) - .5) * spread, rng.random(n) * 5,
                     rng.random(n) * 5, (rng.random(n) - .5) * 10], 1)


def lidar(rng, n, rho_max=80.0, span=3.6):
    rho = rho_max * rng.random(n) ** 2
    th = (rng.random(n) - .5) * span
    z = rng.normal(-1.2, 0.6, n)
    inten = rng.random(n)
    return np.stack([rho * np.cos(th), rho * np.sin(th), z, inten], 1).astype(np.float32)


def proposals(rng, n, n_obj, extent=75.0):
    ctr = (rng.random((n_obj, 2)) - .5) * 2 * extent
    hd = (rng.random(n_obj) - .5) * 2 * np.pi
    k = rng.integers(0, n_obj, n)
    xy = ctr[k] + rng.normal(0, 0.3, (n, 2))
    wh = np.array([4.5, 2.0]) + rng.normal(0, 1, (n, 2)) * np.array([.2, .1])
    r = hd[k] + rng.normal(0, 0.05, n)
    scores = rng.permutation(n).astype(np.float64) / n + rng.random(n) * 0.1 / n
    return np.concatenate([xy, wh, r[:, None]], 1), scores


SOFT_CASES = [  # tests/golden/make_golden.py SOFT_CASES: (tag, n, generator, method, iou_threshold, score_threshold, supression_param)
    ("c1_lin", 1000, "boxes", "linear", 0.3, 0.2, 1.0), ("c1_gau", 1000, "boxes", "gaussian", 0.3, 0.2, 0.5),
    ("c1_lin0", 1000, "boxes", "linear", 0.0, 0.0, 2.0), ("c1_gau_box", 1000, "boxes", "gaussian", 0.25, 0.3, 0.3),
    ("p_lin", 4097, "proposals", "linear", 0.3, 0.1, 1.0), ("p_gau", 4097, "proposals", "gaussian", 0.5, 0.05, 0.5),
]
SOFT_TEST6 = (np.array([[1, 1, 2 - 1e-2, 2 - 1e-2, 0], [2, 2, 2 - 1e-2, 2 - 1e-2, 1e-3], [3, 3, 2 - 1e-2, 2 - 1e-2, 2e-3], [3, 1, 1, 2, 3e-3],
                        [4, 2, 1, 2, 4e-3], [5, 3, 1, 2, 5e-3]], np.float64), np.array([0.5, 0.3, 0.4, 0.4, 0.2, 0.1], np.float64))


def soft_inputs(n, gen):
    """inputs of the soft-NMS fixtures (tests/golden/make_golden.py soft_inputs): regenerated from the seed"""
    rng = np.random.default_rng(1234 + n)
    if gen == "boxes":
        return gen_boxes(rng, n), rng.random(n)
    return proposals(rng, n, max(n // 25, 1))


# inputs of the comparisons with the reference's own code in test_oracle_pinned.py; tests/golden/make_golden.py write_live_ref
# stores the outputs on them in live_ref.npz
LIVE_VOXEL = ([0, 70.4, -40, 40, -3, 1], [352, 400, 40], dict(max_points=3, max_points_filter="trim", max_voxels=900, max_voxels_filter="trim"))


def live_iou_nms_voxel_inputs():
    rng = np.random.default_rng(11)
    A, B = gen_boxes(rng, 300), gen_boxes(rng, 200)
    s = rng.random(300)
    return A, B, s, lidar(rng, 4000)


def live_dist3d_inputs():
    rng = np.random.default_rng(8)
    mk = lambda n: np.concatenate([(rng.random((n, 2)) - .5) * 10, rng.normal(0, 0.5, (n, 1)), rng.random((n, 3)) * 4 + .3,  # noqa: E731
                                   (rng.random((n, 1)) - .5) * 10], 1).astype(np.float32)
    a, b = mk(150), mk(120)
    return a, b, ((rng.random((200, 3)) - .5) * 8).astype(np.float32)


def live_pdist_inputs():
    rng = np.random.default_rng(3)
    pts, bx = (rng.random((2000, 2)) - .5) * 14, gen_boxes(rng, 50)
    p3, b3 = (rng.random((500, 3)) - .5) * 10, np.concatenate([gen_boxes(rng, 20)[:, :2], rng.random((20, 1)), rng.random((20, 3)) * 4 + .2, rng.random((20, 1)) * 6], 1)
    return pts, bx, p3, b3


def assert_pinned(g, name, a):
    """`a` equals golden entry `name` bit for bit: the stored array, or for a large one (make_golden.py pin) the SHA-256 of its bytes,
    after a stored sample of its values that shows where they differ"""
    a = np.ascontiguousarray(a)
    if name in g.files:
        exp = g[name]
        assert a.dtype == exp.dtype and a.shape == exp.shape and np.array_equal(a, exp), name
        return
    idx, val = g[name + ".idx"], g[name + ".val"]
    assert a.dtype == val.dtype and a.shape == tuple(g[name + ".shape"]), (name, a.dtype, a.shape)
    got = a.reshape(-1)[idx]
    bad = np.flatnonzero(got != val)
    assert not len(bad), (name, idx[bad[:5]], got[bad[:5]], val[bad[:5]])
    assert hashlib.sha256(a.tobytes()).hexdigest() == str(g[name + ".sha256"]), name
