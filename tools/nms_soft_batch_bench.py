#!/usr/bin/env python
"""Frame-batched soft-NMS against one box2d_nms call per frame, on the frames of BASELINE config 5 (64 x proposals(900 + f, 4096, 160),
as bench.py's bench_c5 builds them), fp64, rotated boxes, gaussian (iou 0.3, score 0.2, param 0.5: bench.py's soft setting) and
linear (param 1.0).  Every form is timed with CUDA events, one event pair per step, a 256 MB memset between steps (the frames' working
set fits L2), the forms alternating in one process after a warm-up.  Rows: the 64-frame batch, the loop of 64 single-frame calls, and a
batch of one frame against one box2d_nms call on that frame.  Also written: kept counts, whether every batched mask equals the
per-frame one, the GPU's name and power limit, and the kernel times of one batched call (torch.profiler, a run of its own).

    python tools/nms_soft_batch_bench.py --out profiles/r3_nms_soft_batch.json [--steps 3] [--frames 64]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch
from torch.profiler import profile, ProfilerActivity

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from bench import proposals  # noqa: E402
from d3d_b200.box import box2d_nms, box2d_nms_batch  # noqa: E402

SETTINGS = {"gaussian": dict(iou_threshold=0.3, score_threshold=0.2, supression_param=0.5),
            "linear": dict(iou_threshold=0.3, score_threshold=0.2, supression_param=1.0)}


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:   # the name from torch is still recorded
        q = f"nvidia-smi unavailable ({e})"
    return dict(torch_name=torch.cuda.get_device_name(0), nvidia_smi=q)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=64)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    F, NP = args.frames, 4096
    props = [proposals(900 + f, NP, 160) for f in range(F)]
    pb = torch.cat([torch.from_numpy(b) for b, _ in props]).cuda()
    ps = torch.cat([torch.from_numpy(s) for _, s in props]).cuda()
    offs = torch.arange(F + 1, dtype=torch.int64) * NP
    offs_dev = offs.cuda()
    one_b, one_s = pb[:NP].contiguous(), ps[:NP].contiguous()
    one_off = torch.tensor([0, NP], dtype=torch.int64)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    result = dict(workload=f"{F} frames x proposals(900 + f, {NP}, 160), fp64, rbox", gpu=gpu_info(),
                  timing="CUDA events per step, 256 MB memset between steps, forms alternating", steps=args.steps, warmup=args.warmup)
    for method, kw in SETTINGS.items():
        forms = {
            "batch": lambda: box2d_nms_batch(pb, ps, offs, iou_method="rbox", offsets_dev=offs_dev, supression_method=method, **kw),
            "per_frame_loop": lambda: torch.cat([box2d_nms(pb[f * NP:(f + 1) * NP], ps[f * NP:(f + 1) * NP], "rbox", method, **kw)
                                                 for f in range(F)]),
            "batch_of_one": lambda: box2d_nms_batch(one_b, one_s, one_off, iou_method="rbox", supression_method=method, **kw),
            "single_call": lambda: box2d_nms(one_b, one_s, "rbox", method, **kw),
        }
        out = {k: None for k in forms}
        for _ in range(args.warmup):
            for k, fn in forms.items():
                out[k] = fn()
        torch.cuda.synchronize()
        ms = {k: [] for k in forms}
        for _ in range(args.steps):
            for k, fn in forms.items():
                flush.zero_()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                out[k] = fn()
                e1.record()
                torch.cuda.synchronize()
                ms[k].append(e0.elapsed_time(e1))
        kept = [int(out["batch"][f * NP:(f + 1) * NP].sum()) for f in range(F)]
        row = dict(settings=kw,
                   ms={k: dict(mean=float(np.mean(v)), min=float(np.min(v)), all=[round(x, 3) for x in v]) for k, v in ms.items()},
                   batch_speedup_over_loop=float(np.mean(ms["per_frame_loop"]) / np.mean(ms["batch"])),
                   batch_of_one_over_single_call=float(np.mean(ms["batch_of_one"]) / np.mean(ms["single_call"])),
                   masks_equal=bool(torch.equal(out["batch"], out["per_frame_loop"])),
                   batch_of_one_mask_equal=bool(torch.equal(out["batch_of_one"], out["single_call"])),
                   kept_per_frame=dict(min=min(kept), max=max(kept), mean=float(np.mean(kept)), total=sum(kept)))
        # kernel times of one batched call in a run of its own (the profiler slows the host, not the kernels)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            forms["batch"]()
            torch.cuda.synchronize()
        kern = {}
        for ev in prof.key_averages():
            for tag in ("nmsb_sort_kernel", "nmsbs_cand_kernel", "nmsbs_walk_kernel"):
                if tag in ev.key:
                    kern[tag] = kern.get(tag, 0.0) + ev.self_device_time_total
        row["kernels_us_one_batch_call"] = {k: round(v, 1) for k, v in kern.items()}
        result[method] = row
        print(method, json.dumps({k: row[k] for k in ("batch_speedup_over_loop", "batch_of_one_over_single_call", "masks_equal",
                                                     "batch_of_one_mask_equal")}), {k: round(v["mean"], 3) for k, v in row["ms"].items()},
              flush=True)
    text = json.dumps(result, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
