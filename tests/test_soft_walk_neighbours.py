"""CPU restatement of the walk of the batched soft-NMS (nmsbs_walk_kernel, d3d_b200/csrc/nms.cu) against the reference's walk
(nms.cpp:33-94, as orc_nms2d restates it): after a kept box has decayed every box behind it whose IoU exceeds the threshold, the
positions between it and the last suppressed box S are re-sorted with a stable insertion sort.  The batched walk changes two things:

* a kept box decays only the boxes of its candidate list that are behind it -- the list is a superset of the boxes whose IoU with it
  can exceed the threshold, in either order of the pair, and holds no IoU values (the walk evaluates iou(visited, later) itself);
* S is a running value, the larger of the previous S and the positions of the boxes suppressed at this step; when a decay lifts a
  suppressed box back over the score threshold (negative scores), S is found again by a scan.

Both must give the reference's order, S and keep mask at every step."""
import zlib

import numpy as np
import pytest


def coef(v, method, param):
    return 1.0 - v ** param if method == "linear" else np.exp(-v * v / param)


def resort(order, sc, sup, _i, S):
    """nms.cpp:74-94 (orc_nms2d): insertion sort of positions (_i, S); position S and the ones behind it stay"""
    for _j in range(S - 1, _i, -1):
        j, _k = order[_j], _j + 1
        while _k < S and (sup[j] or sc[order[_k]] > sc[j]):
            order[_k - 1] = order[_k]
            _k += 1
        order[_k - 1] = j


def reference_walk(scores, iou, thr, sthr, method, param):
    n = len(scores)
    sc = scores.copy()
    order = list(np.argsort(-sc, kind="stable"))     # stable descending: ties keep the lower index first
    sup = ~(sc > sthr)                               # reference CUDA score rule
    trace, seen = [], dict(redecayed=0, revived=0, mid_S=0)
    for _i in range(n):
        i = order[_i]
        if sup[i]:
            break
        for _j in range(_i + 1, n):
            j = order[_j]
            v = iou[i, j]
            if v > thr:
                was = sup[j]
                sc[j] *= coef(v, method, param)
                sup[j] = sc[j] < sthr
                seen["redecayed"] += int(was)
                seen["revived"] += int(was and not sup[j])
        S = n - 1
        while S > _i and not sup[order[S]]:
            S -= 1
        seen["mid_S"] += int(_i + 1 < S < n - 1)
        resort(order, sc, sup, _i, S)
        trace.append((S, tuple(order)))
    return sup, trace, seen


def neighbour_walk(scores, iou, nbrs, thr, sthr, method, param):
    n = len(scores)
    sc = scores.copy()
    order = list(np.argsort(-sc, kind="stable"))
    sup = ~(sc > sthr)
    pos = np.empty(n, int)
    pos[order] = np.arange(n)
    s_run = max([q for q in range(n) if sup[order[q]]], default=0)
    trace = []
    for _i in range(n):
        i = order[_i]
        if sup[i]:
            break
        s_new, revived = _i, False
        for j in nbrs[i]:
            q = pos[j]
            if q <= _i:
                continue
            v = iou[i, j]
            if v > thr:
                was = sup[j]
                sc[j] *= coef(v, method, param)
                sup[j] = sc[j] < sthr
                revived |= bool(was and not sup[j])
            if sup[j]:
                s_new = max(s_new, q)
        if revived:
            S = max([q for q in range(_i + 1, n) if sup[order[q]]], default=_i)
        else:
            S = max(s_new, s_run)
        s_run = S
        resort(order, sc, sup, _i, S)
        pos[order] = np.arange(n)
        trace.append((S, tuple(order)))
    return sup, trace


def frame(rng, n, kind, thr):
    """scores, an IoU matrix (not symmetric: the clip is evaluated with the visited box first) and candidate lists that hold every pair
    above the threshold in either order plus pairs below it"""
    xy = rng.random((n, 2)) * (4.0 if kind == "crowd" else 10.0)
    near = np.hypot(*(xy[:, None, :] - xy[None, :, :]).transpose(2, 0, 1)) < 1.5
    if kind == "chain":                              # box k overlaps k + 1 only: decays run down the whole frame
        near = np.abs(np.arange(n)[:, None] - np.arange(n)[None, :]) == 1
    np.fill_diagonal(near, False)
    hi = thr + (1.0 - thr) * rng.random((n, n))
    lo = thr * rng.random((n, n))
    lo[rng.random((n, n)) < 0.1] = thr               # exactly at the threshold: not above it
    iou = np.where(near & (rng.random((n, n)) < 0.8), hi, lo)
    iou[~near] = lo[~near]
    extra = rng.random((n, n)) < 0.05                # candidates whose IoU stays below the threshold
    cand = near | extra | extra.T
    np.fill_diagonal(cand, False)
    nbrs = [list(rng.permutation(np.flatnonzero(cand[k]))) for k in range(n)]
    if kind == "ties":
        scores = rng.integers(1, 6, n) / 5.0
    elif kind == "negative":                         # scores below zero: a decay can lift a suppressed box back over the threshold
        scores = rng.random(n) * 2.0 - 1.0
    elif kind == "midS":                             # every score above the threshold of the case (0.45)
        scores = 0.5 + 0.5 * rng.random(n)
    else:
        scores = rng.random(n)
    if kind == "chain":
        scores = np.sort(scores)[::-1].copy()        # chain order = score order
    return scores, iou, nbrs


CASES = [  # (kind, method, param, iou threshold, score threshold, what the case must have met in the reference walk)
    ("midS", "gaussian", 0.5, 0.3, 0.45, "mid_S"),       # no box starts below the score threshold: S starts at none, then grows
    ("midS", "linear", 1.0, 0.2, 0.45, "mid_S"),
    ("chain", "linear", 0.6, 0.1, 0.05, "redecayed"),
    ("chain", "gaussian", 0.3, 0.0, -0.5, None),
    ("ties", "gaussian", 0.5, 0.3, 0.2, "redecayed"),
    ("ties", "linear", 2.0, 0.0, 0.1, "redecayed"),
    ("crowd", "gaussian", 0.1, 0.2, 0.3, "redecayed"),   # dense: boxes are decayed again after they are suppressed
    ("crowd", "linear", 0.5, 0.4, 0.05, "redecayed"),
    ("negative", "linear", 1.0, 0.3, -0.3, "revived"),
    ("negative", "gaussian", 0.4, 0.1, -0.6, "revived"),
]


@pytest.mark.parametrize("kind,method,param,thr,sthr,needs", CASES)
def test_neighbour_decay_and_running_S_follow_the_reference_walk(kind, method, param, thr, sthr, needs):
    rng = np.random.default_rng(zlib.crc32(f"{kind}/{method}".encode()))
    met = 0
    for _ in range(25):
        n = int(rng.integers(1, 90))
        scores, iou, nbrs = frame(rng, n, kind, thr)
        sup_r, tr_r, seen = reference_walk(scores, iou, thr, sthr, method, param)
        sup_n, tr_n = neighbour_walk(scores, iou, nbrs, thr, sthr, method, param)
        assert len(tr_r) == len(tr_n)
        for t, (a, b) in enumerate(zip(tr_r, tr_n)):
            assert a[0] == b[0], (kind, n, "S", t)
            assert a[1] == b[1], (kind, n, "order", t)
        assert np.array_equal(sup_r, sup_n), (kind, n)
        met += seen[needs] if needs else 1
    assert met, (kind, needs)
