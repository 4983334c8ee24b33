"""Detection-evaluator matching over a validation set: the per-frame Python loop of box3d_iou_distance + match_greedy against the
frame-batched box3d_iou_distance_batch + match_greedy_batch.

Workload (seeded): 6000 frames; per frame Poisson(40) ground-truth boxes and Poisson(150) detections, a third of them on a ground-truth
box, 3 classes; all inputs already on the GPU.  Each timed pass computes the rotated distance matrices and the matching for T threshold
sets (T = 1 and T = 40, the evaluator's score thresholds), timed with CUDA events and ended by a device synchronise, after one warm-up
pass.  Prints one JSON line with the GPU name and power limit, the times and whether the two paths give equal outputs.

    python tools/eval_batch_bench.py [--frames 6000] [--repeats 3]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from d3d_b200.box import box3d_iou_distance, box3d_iou_distance_batch, match_greedy, match_greedy_batch  # noqa: E402


def workload(nframes, seed=0):
    rng = np.random.default_rng(seed)

    def boxes(n):
        return np.stack([(rng.random(n) - .5) * 100, (rng.random(n) - .5) * 100, rng.normal(-1, 0.5, n), 3.5 + rng.random(n) * 2,
                         1.5 + rng.random(n), 1.4 + rng.random(n) * 0.6, (rng.random(n) - .5) * 7], 1).astype(np.float32)
    ng, nd = rng.poisson(40, nframes), rng.poisson(150, nframes)
    gts, dts = [], []
    for g, d in zip(ng, nd):
        gt, dt = boxes(g), boxes(d)
        k = min(g, d // 3)
        if k:
            dt[:k] = gt[rng.integers(0, g, k)] + rng.normal(0, 0.2, (k, 7)).astype(np.float32)
        gts.append(gt)
        dts.append(dt)
    scores = [rng.random(d) for d in nd]
    dtags = [rng.integers(0, 3, d).astype(np.int32) for d in nd]
    gtags = [rng.integers(0, 3, g).astype(np.int32) for g in ng]
    return dts, gts, scores, dtags, gtags


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        name, power = out.stdout.strip().splitlines()[0].split(", ")
        return name, power
    except Exception as e:   # the numbers are still printed; where they come from is then unknown
        return torch.cuda.get_device_name(0), f"unknown ({e})"


def timed(fn, repeats):
    fn()
    torch.cuda.synchronize()
    times, out = [], None
    for _ in range(repeats):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out = fn()
        b.record()
        torch.cuda.synchronize()
        times.append(a.elapsed_time(b))
    return times, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=6000)
    ap.add_argument("--repeats", type=int, default=3)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "the benchmark needs a CUDA device"
    dev = torch.device("cuda:0")
    dts, gts, scores, dtags, gtags = workload(args.frames)
    t = lambda xs: [torch.from_numpy(x).to(dev) for x in xs]  # noqa: E731
    dl, gl, sl, dtl, gtl = t(dts), t(gts), t(scores), t(dtags), t(gtags)
    so, go = np.cumsum([0] + [len(x) for x in dts]), np.cumsum([0] + [len(x) for x in gts])
    dp, gp, sp = torch.cat(dl), torch.cat(gl), torch.cat(sl)
    dtp, gtp = torch.cat(dtl), torch.cat(gtl)
    so_t, go_t = torch.from_numpy(so), torch.from_numpy(go)
    thr_all = torch.from_numpy(np.stack([np.array([0.3, 0.5, 0.5]) + x for x in np.linspace(0.0, 0.65, 40)]).astype(np.float32)).to(dev)
    name, power = gpu_info()
    results = []
    for T in (1, 40):
        thr = thr_all[:T]

        def loop():
            ds, sa, da = [], [], []
            for f in range(args.frames):
                d = box3d_iou_distance(dl[f], gl[f], "riou")
                a, b = match_greedy(d, sl[f], dtl[f], gtl[f], thr)
                ds.append(d.reshape(-1))
                sa.append(a)
                da.append(b)
            return torch.cat(ds), torch.cat(sa, 1), torch.cat(da, 1)

        def batch():
            flat, doff = box3d_iou_distance_batch(dp, gp, so_t, go_t, metric="riou")
            a, b = match_greedy_batch((flat, doff), sp, dtp, gtp, thr, so_t, go_t)
            return flat, a, b

        t_loop, o_loop = timed(loop, args.repeats)
        t_batch, o_batch = timed(batch, args.repeats)
        equal = bool(torch.equal(o_loop[0].view(torch.int32), o_batch[0].view(torch.int32)) and torch.equal(o_loop[1], o_batch[1])
                     and torch.equal(o_loop[2], o_batch[2]))
        results.append(dict(T=T, loop_ms=[round(x, 3) for x in t_loop], batch_ms=[round(x, 3) for x in t_batch],
                            speedup=round(min(t_loop) / min(t_batch), 2), outputs_equal=equal, matches=int((o_batch[1] >= 0).sum())))
    print(json.dumps(dict(bench="eval_batch", gpu=name, power_limit=power, frames=args.frames, detections=int(so[-1]), ground_truth=int(go[-1]),
                          classes=3, results=results)))


if __name__ == "__main__":
    main()
