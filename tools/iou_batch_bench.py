"""Differentiable IoU family over a training batch: the per-frame Python loop of box2d_iou against the frame-batched box2d_iou_batch.

Workloads (seeded; every frame has Poisson(40) KITTI-sized ground-truth boxes, 3.5-5.5 x 1.5-2.5 m, any heading, in the
[0, 70.4] x [-40, 40] m PointPillars range):
  roi      16 frames x 512 proposals (region-of-interest targets): proposals jittered around the frame's ground truth and uniform clutter;
  c5       64 frames x 4096 proposals, the same distribution;
  anchors  4 frames x 107 136 anchors: the 216 x 248 PointPillars grid, two headings (0, pi / 2), 3.9 x 1.6 m.
Each workload is timed for "rbox" and "box" forward, and "grbox" / "drbox" forward and forward plus backward of sum(values) into both box
sets; in fp32 (precise=False) and in the default fp64 (precise=True on fp32 inputs).  All inputs are on the GPU before timing; the batch
calls take the per-frame lists.  Each timing is CUDA events around one call ended by a device synchronise, after one warm-up call; best
and median of --repeats.  "equal" is whether the batched values (and gradients) equal the loop's bit for bit; "launches" is
d3d_launch_count per call.  Prints one JSON line with the GPU name and power limit.

--box-kernels instead compares the two layouts of the "box" kernel on each workload: the summed device time of the per-frame loop's
iou2d_kernel (one CTA per row and 1024 columns) against the batch's iou2d_batch_kernel (the frame's (row, 4-column chunk) pairs flattened
over the CTAs), from torch.profiler over --repeats calls each, after a warm-up.  One JSON line as well.

    python tools/iou_batch_bench.py [--workloads roi c5 anchors] [--repeats 5] [--box-kernels]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from d3d_b200 import _cabi  # noqa: E402
from d3d_b200.box import box2d_iou, box2d_iou_batch  # noqa: E402

WORKLOADS = {"roi": (16, 512), "c5": (64, 4096), "anchors": (4, None)}


def ground_truth(rng):
    m = int(rng.poisson(40))
    return np.stack([rng.random(m) * 70.4, (rng.random(m) - .5) * 80, 3.5 + rng.random(m) * 2, 1.5 + rng.random(m),
                     (rng.random(m) - .5) * 2 * np.pi], 1)


def proposals(rng, gt, n):
    """half jittered around the ground truth, half uniform clutter"""
    k = n // 2 if len(gt) else 0
    j = gt[rng.integers(0, max(len(gt), 1), k)] + rng.normal(0, [0.6, 0.6, 0.3, 0.2, 0.3], (k, 5)) if k else np.zeros((0, 5))
    u = np.stack([rng.random(n - k) * 70.4, (rng.random(n - k) - .5) * 80, 3.5 + rng.random(n - k) * 2, 1.5 + rng.random(n - k),
                  (rng.random(n - k) - .5) * 2 * np.pi], 1)
    return np.concatenate([j, u])


def anchors():
    x, y = np.meshgrid((np.arange(216) + .5) * 70.4 / 216, (np.arange(248) + .5) * 80 / 248 - 40, indexing="ij")
    c = np.stack([x.ravel(), y.ravel()], 1)
    return np.concatenate([np.c_[c, np.full((len(c), 3), [3.9, 1.6, 0.0])], np.c_[c, np.full((len(c), 3), [3.9, 1.6, np.pi / 2])]])


def workload(name, seed=0):
    rng = np.random.default_rng(seed)
    nframes, n = WORKLOADS[name]
    b1, b2 = [], []
    for _ in range(nframes):
        gt = ground_truth(rng)
        b1.append((anchors() if n is None else proposals(rng, gt, n)).astype(np.float32))
        b2.append(gt.astype(np.float32))
    return b1, b2


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        name, power = out.stdout.strip().splitlines()[0].split(", ")
        return name, power
    except Exception as e:   # the numbers are still printed; where they come from is then unknown
        return torch.cuda.get_device_name(0), f"unknown ({e})"


def timed(fn, repeats):
    out = fn()
    torch.cuda.synchronize()
    c0 = _cabi.launch_count()
    out = fn()
    torch.cuda.synchronize()
    launches = _cabi.launch_count() - c0
    times = []
    for _ in range(repeats):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out = fn()
        b.record()
        torch.cuda.synchronize()
        times.append(a.elapsed_time(b))
    return dict(best_ms=round(min(times), 3), median_ms=round(statistics.median(times), 3), launches=launches), out


def same_bits(xs, ys):
    return all(x.dtype == y.dtype and x.shape == y.shape and torch.equal(x.view(torch.int32 if x.dtype == torch.float32 else torch.int64),
                                                                         y.view(torch.int32 if y.dtype == torch.float32 else torch.int64))
               for x, y in zip(xs, ys))


def run(name, repeats, dev):
    b1, b2 = workload(name)
    l1, l2 = [torch.from_numpy(b).to(dev) for b in b1], [torch.from_numpy(b).to(dev) for b in b2]
    res = dict(workload=name, frames=len(b1), boxes1=sum(map(len, b1)), boxes2=sum(map(len, b2)), pairs=sum(len(a) * len(b) for a, b in zip(b1, b2)))
    g1, g2 = [x.clone().requires_grad_(True) for x in l1], [x.clone().requires_grad_(True) for x in l2]

    def fwd_bwd(method, precise, batched):
        for x in g1 + g2:
            x.grad = None
        vs = box2d_iou_batch(g1, g2, method=method, precise=precise) if batched else [box2d_iou(a, b, method, precise) for a, b in zip(g1, g2)]
        sum(v.sum() for v in vs).backward()
        return [x.grad.clone() for x in g1 + g2]

    for precise, tag in ((False, "f32"), (True, "f64")):
        for method in ("rbox", "box", "grbox", "drbox"):
            t_loop, v_loop = timed(lambda: [box2d_iou(a, b, method, precise) for a, b in zip(l1, l2)], repeats)
            t_batch, v_batch = timed(lambda: box2d_iou_batch(l1, l2, method=method, precise=precise), repeats)
            res[f"{method}_{tag}_forward"] = dict(loop=t_loop, batch=t_batch, speedup=round(t_loop["best_ms"] / t_batch["best_ms"], 2),
                                                  equal=same_bits(v_loop, v_batch))
            del v_loop, v_batch
            if method in ("grbox", "drbox"):
                t_loop, gr_loop = timed(lambda: fwd_bwd(method, precise, False), repeats)
                t_batch, gr_batch = timed(lambda: fwd_bwd(method, precise, True), repeats)
                res[f"{method}_{tag}_forward_backward"] = dict(loop=t_loop, batch=t_batch, speedup=round(t_loop["best_ms"] / t_batch["best_ms"], 2),
                                                               equal=same_bits(gr_loop, gr_batch))
    return res


def box_kernels(name, repeats, dev):
    from torch.profiler import ProfilerActivity, profile
    b1, b2 = workload(name)
    l1, l2 = [torch.from_numpy(b).to(dev) for b in b1], [torch.from_numpy(b).to(dev) for b in b2]
    res = dict(workload=name, frames=len(b1))
    for precise, tag in ((False, "f32"), (True, "f64")):
        loop = lambda: [box2d_iou(a, b, "box", precise) for a, b in zip(l1, l2)]  # noqa: E731
        batch = lambda: box2d_iou_batch(l1, l2, method="box", precise=precise)  # noqa: E731
        loop(), batch()
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(repeats):
                loop()
                batch()
            torch.cuda.synchronize()
        us = {}
        for e in prof.key_averages():
            for k in ("iou2d_kernel", "iou2d_batch_kernel"):
                if f"::{k}<" in e.key:
                    us[k] = us.get(k, 0.0) + getattr(e, "device_time_total", getattr(e, "cuda_time_total", 0.0)) / repeats
        res[tag] = dict(loop_iou2d_kernel_us=round(us.get("iou2d_kernel", 0.0), 1), batch_iou2d_batch_kernel_us=round(us.get("iou2d_batch_kernel", 0.0), 1))
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", nargs="+", default=list(WORKLOADS), choices=list(WORKLOADS))
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--box-kernels", action="store_true", help="compare the device time of the two \"box\" kernel layouts instead")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "the benchmark needs a CUDA device"
    assert args.repeats >= 3
    dev = torch.device("cuda:0")
    name, power = gpu_info()
    if args.box_kernels:
        results = [box_kernels(w, args.repeats, dev) for w in args.workloads]
        print(json.dumps(dict(bench="iou_batch_box_kernels", gpu=name, power_limit=power, repeats=args.repeats, results=results)))
        return
    results = [run(w, args.repeats, dev) for w in args.workloads]
    equal = all(v["equal"] for r in results for v in r.values() if isinstance(v, dict))
    print(json.dumps(dict(bench="iou_batch", gpu=name, power_limit=power, repeats=args.repeats, equal=equal, results=results)))


if __name__ == "__main__":
    main()
