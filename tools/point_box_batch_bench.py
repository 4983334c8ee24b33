"""Point <-> box operators over a training batch: the per-frame Python loop of box3dp_crop / box3dr_pdist against the frame-batched
box3dp_crop_batch / box3dr_pdist_batch.

Workload (seeded): 16 and 64 frames; each frame is a C2 lidar cloud (bench.lidar: 120 000 points, xyz float32) with Poisson(40)
KITTI-sized 3-D boxes (3.5-5.5 x 1.5-2.5 x 1.4-2.0 m, any heading) centred on cloud points; all inputs already on the GPU, the batch
calls take the per-frame lists.  Timed: box3dp_crop (fp32 mask), box3dr_pdist forward, and forward plus backward of sum(distances)
into points and boxes.  Each timing is CUDA events around one pass ended by a device synchronise, after one warm-up pass; best and
median of --repeats passes.  Prints one JSON line with the GPU name and power limit, the times and whether the batched outputs equal the
loop's (masks and distances bit for bit, gradients to a relative 1e-4).  The masks of a 16-frame batch (~77 MB) fit in the 126 MB L2;
the distances and the 64-frame masks do not.

    python tools/point_box_batch_bench.py [--frames 16 64] [--repeats 5]
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
import bench  # noqa: E402
from d3d_b200.box import box3dp_crop, box3dp_crop_batch, box3dr_pdist, box3dr_pdist_batch  # noqa: E402

L2_BYTES = 126 * 2 ** 20


def workload(nframes, seed=0):
    rng = np.random.default_rng(seed)
    pts, boxes = [], []
    for f in range(nframes):
        p = np.ascontiguousarray(bench.lidar(seed * 1000 + f)[:, :3])
        m = int(rng.poisson(40))
        c = p[rng.integers(0, len(p), m)]
        b = np.concatenate([c, np.stack([3.5 + rng.random(m) * 2, 1.5 + rng.random(m), 1.4 + rng.random(m) * 0.6,
                                         (rng.random(m) - .5) * 2 * np.pi], 1)], 1).astype(np.float32)
        pts.append(p)
        boxes.append(b)
    return pts, boxes


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
    times = []
    for _ in range(repeats):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out = fn()
        b.record()
        torch.cuda.synchronize()
        times.append(a.elapsed_time(b))
    return dict(best_ms=round(min(times), 3), median_ms=round(statistics.median(times), 3)), out


def rel(a, b):
    return float((a.double() - b.double()).abs().max() / max(1.0, float(b.double().abs().max())))


def run(nframes, repeats, dev):
    pts, boxes = workload(nframes)
    pl = [torch.from_numpy(p).to(dev) for p in pts]
    bl = [torch.from_numpy(b).to(dev) for b in boxes]
    pairs = sum(len(p) * len(b) for p, b in zip(pts, boxes))
    res = dict(frames=nframes, points=sum(len(p) for p in pts), boxes=sum(len(b) for b in boxes), pairs=pairs,
               mask_bytes=pairs, mask_fits_l2=pairs < L2_BYTES, dist_bytes=4 * pairs)

    t_loop, m_loop = timed(lambda: [box3dp_crop(p, b) for p, b in zip(pl, bl)], repeats)
    t_batch, m_batch = timed(lambda: box3dp_crop_batch(pl, bl), repeats)
    res["crop"] = dict(loop=t_loop, batch=t_batch, speedup=round(t_loop["best_ms"] / t_batch["best_ms"], 2),
                       equal=all(torch.equal(x, y) for x, y in zip(m_loop, m_batch)))
    del m_loop, m_batch

    t_loop, d_loop = timed(lambda: [box3dr_pdist(p, b) for p, b in zip(pl, bl)], repeats)
    t_batch, d_batch = timed(lambda: box3dr_pdist_batch(pl, bl), repeats)
    res["pdist_forward"] = dict(loop=t_loop, batch=t_batch, speedup=round(t_loop["best_ms"] / t_batch["best_ms"], 2),
                                equal=all(torch.equal(x.view(torch.int32), y.view(torch.int32)) for x, y in zip(d_loop, d_batch)))
    del d_loop, d_batch

    gl = [p.clone().requires_grad_(True) for p in pl]
    hl = [b.clone().requires_grad_(True) for b in bl]

    def fwd_bwd(batched):
        for x in gl + hl:
            x.grad = None
        ds = box3dr_pdist_batch(gl, hl) if batched else [box3dr_pdist(p, b) for p, b in zip(gl, hl)]
        sum(d.sum() for d in ds).backward()
        return [x.grad.clone() for x in gl + hl]
    t_loop, g_loop = timed(lambda: fwd_bwd(False), repeats)
    t_batch, g_batch = timed(lambda: fwd_bwd(True), repeats)
    err = max(rel(x, y) for x, y in zip(g_batch, g_loop))
    res["pdist_forward_backward"] = dict(loop=t_loop, batch=t_batch, speedup=round(t_loop["best_ms"] / t_batch["best_ms"], 2),
                                         grad_rel_err=err, equal=err <= 1e-4)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, nargs="+", default=[16, 64])
    ap.add_argument("--repeats", type=int, default=5)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "the benchmark needs a CUDA device"
    assert args.repeats >= 3
    dev = torch.device("cuda:0")
    name, power = gpu_info()
    results = [run(f, args.repeats, dev) for f in args.frames]
    equal = all(r[k]["equal"] for r in results for k in ("crop", "pdist_forward", "pdist_forward_backward"))
    print(json.dumps(dict(bench="point_box_batch", gpu=name, power_limit=power, repeats=args.repeats, equal=equal, results=results)))


if __name__ == "__main__":
    main()
