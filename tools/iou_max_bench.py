"""Target assignment without the IoU matrix: the fused max-IoU reduction (box2d_iou_max / box2d_iou_max_batch) against the matrix path it
replaces (box2d_iou_batch or box2d_iou, then torch's max along both axes of every frame's matrix).

Workloads (seeded):
  anchors, roi, c5  the frame-batched workloads of tools/iou_batch_bench.py (same generators): 4 x 107 136 anchors, 16 x 512 and
                    64 x 4096 proposals, each frame against Poisson(40) ground truth; "rbox" and "box", fp32 (precise=False) and the
                    default fp64 (precise=True on fp32 inputs);
  c4                one 100 000 x 100 000 frame of the C4 distribution (bench.py's C1 boxes), fp32, precise=False, "rbox": the matrix
                    alone is 40 GB;
  c4_precise        one 30 000 x 30 000 frame of the same distribution, precise=True, "rbox".
Each path is timed with CUDA events around one call ended by a device synchronise, after one warm-up call; best and median of --repeats.
"equal" is whether the fused outputs equal the matrix path's bit for bit (NaN matches NaN); "launches" is d3d_launch_count per call and
"kernels" every CUDA kernel of one call (torch's max kernels included), from torch.profiler in an untimed call; "peak_gb" is
torch.cuda.max_memory_allocated during one call minus what was allocated before it.  For "rbox", "tflops" counts SURVEY.md 8(d)'s
230 flops per candidate pair (bounding circles overlap, count_candidates_kernel) and 8 per rejected pair over the fused call's best
time, next to the FFMA2 (fp32) / DFMA (fp64) peak bench.py measures with d3d_fma_peak_probe in the same run.  Prints one JSON line with
the GPU name and power limit.

    python tools/iou_max_bench.py [--workloads anchors roi c5 c4 c4_precise] [--repeats 5]
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
import iou_batch_bench as IB  # noqa: E402
from d3d_b200 import _cabi  # noqa: E402
from d3d_b200.box import box2d_iou, box2d_iou_batch, box2d_iou_max, box2d_iou_max_batch  # noqa: E402

SINGLE = {"c4": (100_000, False), "c4_precise": (30_000, True)}
WORKLOADS = list(IB.WORKLOADS) + list(SINGLE)


def reduce_matrix(v):
    """torch.max along both axes; (0, -1) where the other side is empty, as the fused path gives it"""
    n, m = v.shape
    if n and m:
        (m1, i1), (m2, i2) = v.max(1), v.max(0)
        return m1, i1, m2, i2
    z = lambda k: (torch.zeros(k, dtype=v.dtype, device=v.device), torch.full((k,), -1, dtype=torch.int64, device=v.device))  # noqa: E731
    return z(n) + z(m)


def same(xs, ys):
    for x, y in zip(xs, ys):
        if x.dtype != y.dtype or x.shape != y.shape:
            return False
        if x.is_floating_point():
            nx, ny = torch.isnan(x), torch.isnan(y)
            iv = torch.int32 if x.dtype == torch.float32 else torch.int64
            if not (torch.equal(nx, ny) and torch.equal(x.view(iv)[~nx], y.view(iv)[~ny])):
                return False
        elif not torch.equal(x, y):
            return False
    return True


def peak_gb(fn):
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    out = fn()
    torch.cuda.synchronize()
    del out
    return round((torch.cuda.max_memory_allocated() - base) / 1e9, 3)


def kernels(fn):
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return sum(1 for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and not e.name.startswith(("Memcpy", "Memset")))


def candidates(l1, l2, code):
    """SURVEY.md 8(d) candidate pairs of every frame (bounding circles overlap), with the library's counter"""
    tot = 0
    for a, b in zip(l1, l2):
        if len(a) and len(b):
            dt = torch.float64 if code else torch.float32
            a, b = a.to(dt).contiguous(), b.to(dt).contiguous()
            cnt = torch.zeros(64, dtype=torch.int64, device=a.device)
            ws = _cabi.workspace(_cabi.iou_workspace_bytes(len(a), len(b), code), a.device)
            _cabi.check(_cabi.iou_count_candidates(_cabi.ptr(a), len(a), _cabi.ptr(b), len(b), code, _cabi.ptr(cnt), _cabi.ptr(ws), ws.numel(),
                                                   _cabi.stream_ptr()), "count")
            tot += int(cnt.sum())
    return tot


def measure(fused, matrix, repeats):
    t_fused, v_fused = IB.timed(fused, repeats)
    t_matrix, v_matrix = IB.timed(matrix, repeats)
    eq = all(same(a, b) for a, b in zip(v_fused, v_matrix))
    del v_fused, v_matrix
    torch.cuda.empty_cache()
    t_fused.update(kernels=kernels(fused), peak_gb=peak_gb(fused))
    t_matrix.update(kernels=kernels(matrix), peak_gb=peak_gb(matrix))
    torch.cuda.empty_cache()
    return dict(fused=t_fused, matrix=t_matrix, speedup=round(t_matrix["best_ms"] / t_fused["best_ms"], 2), equal=eq)


def run(name, repeats, dev, peaks):
    if name in SINGLE:
        n, precise = SINGLE[name]
        rng = np.random.default_rng(3)
        l1, l2 = [torch.from_numpy(bench.gen_boxes(rng, n).astype(np.float32)).to(dev)], [torch.from_numpy(bench.gen_boxes(rng, n).astype(np.float32)).to(dev)]
        cases = [("rbox", precise)]
    else:
        b1, b2 = IB.workload(name)
        l1, l2 = [torch.from_numpy(b).to(dev) for b in b1], [torch.from_numpy(b).to(dev) for b in b2]
        cases = [(m, p) for p in (False, True) for m in ("rbox", "box")]
    pairs = sum(len(a) * len(b) for a, b in zip(l1, l2))
    res = dict(workload=name, frames=len(l1), boxes1=sum(map(len, l1)), boxes2=sum(map(len, l2)), pairs=pairs)
    for method, precise in cases:
        if name in SINGLE:
            fused = lambda: [box2d_iou_max(l1[0], l2[0], method, precise)]  # noqa: E731
            matrix = lambda: [reduce_matrix(box2d_iou(l1[0], l2[0], method, precise))]  # noqa: E731
        else:
            fused = lambda: box2d_iou_max_batch(l1, l2, method=method, precise=precise)  # noqa: E731
            matrix = lambda: [reduce_matrix(v) for v in box2d_iou_batch(l1, l2, method=method, precise=precise)]  # noqa: E731
        r = measure(fused, matrix, repeats)
        code = 1 if precise else 0
        r["pairs_per_s"] = pairs / (r["fused"]["best_ms"] * 1e-3)
        if method == "rbox":
            cand = candidates(l1, l2, code)
            tf = (cand * bench.W_CAND + (pairs - cand) * bench.W_REJ) / (r["fused"]["best_ms"] * 1e-3) / 1e12
            r.update(candidate_fraction=round(cand / pairs, 4), tflops=round(tf, 2), peak_tflops=round(peaks[code], 2), frac_of_peak=round(tf / peaks[code], 3))
        res[f"{method}_{'f64' if precise else 'f32'}"] = r
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", nargs="+", default=WORKLOADS, choices=WORKLOADS)
    ap.add_argument("--repeats", type=int, default=5)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "the benchmark needs a CUDA device"
    assert args.repeats >= 5
    dev = torch.device("cuda:0")
    name, power = IB.gpu_info()
    peaks = {0: bench.fma_peak(0), 1: bench.fma_peak(1)}
    results = [run(w, args.repeats, dev, peaks) for w in args.workloads]
    equal = all(v["equal"] for r in results for v in r.values() if isinstance(v, dict))
    print(json.dumps(dict(bench="iou_max", gpu=name, power_limit=power, repeats=args.repeats, equal=equal, results=results)))


if __name__ == "__main__":
    main()
