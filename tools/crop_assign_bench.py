"""Fused point-in-box reductions (box2dr_crop_assign / box3dp_crop_assign[_batch]) against the mask call plus the torch reductions
(torch.where(mask.any(0), mask.to(torch.uint8).argmax(0), -1) and mask.sum(1) per frame).

Workloads (seeded, all inputs already on the GPU):
  gt_batch      point_box_batch_bench.workload(16) and (64): C2 clouds (120 000 points) with Poisson(40) KITTI-sized 3-D boxes, the
                per-frame lists into box3dp_crop_assign_batch vs box3dp_crop_batch + reductions (tile path).
  proposals     one frame, 180 000 lidar points x 4096 proposals (bench.lidar(300) / bench.proposals(300, 4096, 2048)), fp32:
                box2dr_crop_assign (grid path) vs box2dr_crop + reductions; the fused call is also timed with each back end forced.
  crossover     180 000 points x M proposals for M around the 64 M-pair grid threshold, the fused call with each back end forced.
  proposals_3d  16 frames x (C2 cloud, 4096 proposals made 3-D with z = -1, lz = 1.6): box3dp_crop_assign_batch vs box3dp_crop_batch +
                reductions (every frame is above the threshold: one single-frame grid-path call each); torch.cuda.max_memory_allocated
                above the inputs for both.
Each timing is CUDA events around one pass ended by a device synchronise, after one warm-up pass; best and median of --repeats passes.
Prints one JSON line with the GPU name and power limit and whether the fused outputs equal the reductions of the mask.

    python tools/crop_assign_bench.py [--repeats 5]
"""
import argparse
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import bench  # noqa: E402
from point_box_batch_bench import gpu_info, timed, workload  # noqa: E402
from d3d_b200 import _cabi  # noqa: E402
from d3d_b200.box import box2dr_crop, box2dr_crop_assign, box3dp_crop_assign_batch, box3dp_crop_batch  # noqa: E402


def reduce(mask):
    return torch.where(mask.any(0), mask.to(torch.uint8).argmax(0), -1), mask.sum(1)


def equal(fused, masked):
    return all(torch.equal(a, b) for x, y in zip(fused, masked) for a, b in zip(x, y))


def peak_bytes(fn):
    """bytes allocated by one call above what was allocated before it"""
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    out = fn()
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    del out
    return peak


def compare(fused_fn, mask_fn, repeats):
    t_f, o_f = timed(fused_fn, repeats)
    t_m, o_m = timed(mask_fn, repeats)
    return dict(fused=t_f, mask_and_reduce=t_m, speedup=round(t_m["best_ms"] / t_f["best_ms"], 2), equal=equal(o_f, o_m))


def forced(path, fn, repeats):
    _cabi.tuning_set("D3D_B200_CROP_PATH", {"brute": 1, "grid": 2}[path])
    try:
        return timed(fn, repeats)
    finally:
        _cabi.tuning_set("D3D_B200_CROP_PATH", None)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=5)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "the benchmark needs a CUDA device"
    assert args.repeats >= 3
    dev = torch.device("cuda:0")
    name, power = gpu_info()
    res = {}

    for nf in (16, 64):
        pts, boxes = workload(nf)
        pl, bl = [torch.from_numpy(p).to(dev) for p in pts], [torch.from_numpy(b).to(dev) for b in boxes]
        r = compare(lambda: box3dp_crop_assign_batch(pl, bl), lambda: [reduce(m) for m in box3dp_crop_batch(pl, bl)], args.repeats)
        r.update(frames=nf, points=sum(len(p) for p in pts), boxes=sum(len(b) for b in boxes), mask_bytes=sum(len(p) * len(b) for p, b in zip(pts, boxes)))
        res[f"gt_batch_{nf}"] = r
        del pl, bl

    P = torch.from_numpy(bench.lidar(300, 180_000)[:, :2].copy()).to(dev)
    B = torch.from_numpy(bench.proposals(300, 4096, 2048)[0].astype(np.float32)).to(dev)
    r = compare(lambda: [box2dr_crop_assign(P, B)], lambda: [reduce(box2dr_crop(P, B))], args.repeats)
    r.update(points=len(P), boxes=len(B), mask_bytes=len(P) * len(B))
    r["fused_brute"], out_b = forced("brute", lambda: [box2dr_crop_assign(P, B)], args.repeats)
    r["fused_grid"], out_g = forced("grid", lambda: [box2dr_crop_assign(P, B)], args.repeats)
    r["equal"] = r["equal"] and equal(out_b, out_g) and equal(out_b, [reduce(box2dr_crop(P, B))])
    res["proposals"] = r
    del out_b, out_g

    cross = []
    ok = True
    for m in (64, 256, 373, 512, 1024, 4096):
        Bm = B[:m].contiguous()
        tb, ob = forced("brute", lambda: box2dr_crop_assign(P, Bm), args.repeats)
        tg, og = forced("grid", lambda: box2dr_crop_assign(P, Bm), args.repeats)
        ok = ok and equal([ob], [og])
        cross.append(dict(boxes=m, mpairs=round(len(P) * m / 2 ** 20, 1), brute=tb, grid=tg))
    res["crossover"] = dict(points=len(P), grid_min_mpairs=int(_cabi.crop_grid_min_pairs()) // 2 ** 20, sizes=cross, equal=ok)
    del P, B

    pl, bl = [], []
    for f in range(16):
        pl.append(torch.from_numpy(np.ascontiguousarray(bench.lidar(f)[:, :3])).to(dev))
        b2 = bench.proposals(100 + f, 4096, 2048)[0]
        b3 = np.stack([b2[:, 0], b2[:, 1], np.full(len(b2), -1.0), b2[:, 2], b2[:, 3], np.full(len(b2), 1.6), b2[:, 4]], 1)
        bl.append(torch.from_numpy(b3.astype(np.float32)).to(dev))
    r = compare(lambda: box3dp_crop_assign_batch(pl, bl), lambda: [reduce(m) for m in box3dp_crop_batch(pl, bl)], args.repeats)
    r.update(frames=16, points=sum(len(p) for p in pl), boxes=sum(len(b) for b in bl), mask_bytes=sum(len(p) * len(b) for p, b in zip(pl, bl)))
    r["fused_peak_bytes"] = peak_bytes(lambda: box3dp_crop_assign_batch(pl, bl))
    r["mask_and_reduce_peak_bytes"] = peak_bytes(lambda: [reduce(m) for m in box3dp_crop_batch(pl, bl)])
    res["proposals_3d_batch"] = r

    eq = all(v["equal"] for v in res.values())
    print(json.dumps(dict(bench="crop_assign", gpu=name, power_limit=power, repeats=args.repeats, equal=eq, results=res)))


if __name__ == "__main__":
    main()
