#!/usr/bin/env python
"""bench.py -- throughput of the d3d hot path on B200 next to the reference's CPU path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--op all|voxel|iou|nms|scatter|dist3d|crop] [--impl reference] [--dump-outputs DIR]
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W      (N > 1)

One JSON line on rank 0.  BASELINE.json's metric is a triple (rotated-IoU pairs/s, NMS boxes/s, voxelized
points/s); the top-level `metric`/`value` of the line is voxelized points/s on config C2 (configs[1]: the
configuration the tier names for N=1, HBM-bound like the `roofline` contract expects) and the other two
operators are reported with the same keys under `ops` (`ops.iou`: config C4 100k x 100k fp32,
`ops.nms`: config C3 50k proposals fp64).  `--op iou|nms` makes that operator the top-level line.

  value     device-resident inputs, CUDA-event timed, K steps after W warm-ups, max over ranks
  e2e       same metric through the public Python API with HOST tensors (H2D of the inputs and D2H of the
            results inside the timed region)
  roofline  algorithmic bytes (voxel: 16N + 32K + 28V' per frame, SURVEY.md 8(d)) or flops (IoU: 230 per
            candidate pair + 8 per rejected pair) over the CUDA-event time, against the measured peak
  cpu_baseline  the reference's own CPU extension (oracle/_ref, kind "reference") or the C oracle ("port")
            on this box's host cores, bounded sample, rank 0 at N=1 only
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

C2_BOUNDS, C2_SHAPE = [0, 70.4, -40, 40, -3, 1], [1408, 1600, 40]
C2_KW = dict(max_points=5, max_points_filter="trim")
C2_POINTS = 120_000
W_CAND, W_REJ = 230.0, 8.0   # SURVEY.md 8(d): algorithmic FP ops per candidate / rejected pair


# ------------------------------------------------------------------ synthetic inputs (SURVEY.md 8(d), Appendix C)
def lidar(seed, n=C2_POINTS):
    rng = np.random.default_rng(seed)
    rho = 80 * rng.random(n) ** 2
    th = (rng.random(n) - .5) * 3.6
    z = rng.normal(-1.2, 0.6, n)
    inten = rng.random(n)
    return np.stack([rho * np.cos(th), rho * np.sin(th), z, inten], 1).astype(np.float32)


def gen_boxes(rng, n):
    return np.stack([(rng.random(n) - .5) * 10, (rng.random(n) - .5) * 10, rng.random(n) * 5, rng.random(n) * 5,
                     (rng.random(n) - .5) * 10], 1)


def proposals(seed, n=50_000, n_obj=2000, extent=75.0):
    rng = np.random.default_rng(seed)
    ctr = (rng.random((n_obj, 2)) - .5) * 2 * extent
    hd = (rng.random(n_obj) - .5) * 2 * np.pi
    k = rng.integers(0, n_obj, n)
    xy = ctr[k] + rng.normal(0, 0.3, (n, 2))
    wh = np.array([4.5, 2.0]) + rng.normal(0, 1, (n, 2)) * np.array([.2, .1])
    r = hd[k] + rng.normal(0, 0.05, n)
    scores = rng.permutation(n).astype(np.float64) / n + rng.random(n) * 0.1 / n
    return np.concatenate([xy, wh, r[:, None]], 1), scores


# ------------------------------------------------------------------ CPU baseline (reference extension or C oracle)
def _cpu_kind():
    try:
        from oracle import ref as R
        if R.available():
            R._voxel(); R._box()
            return "reference"
    except Exception:
        pass
    return "port"


def _cpu_voxel_frame(seed):
    import torch
    torch.set_num_threads(1)
    pts = lidar(seed)
    kind = _CPU_KIND
    t0 = time.perf_counter()
    if kind == "reference":
        from oracle import ref as R
        R.VoxelGenerator(C2_BOUNDS, C2_SHAPE, **C2_KW)(pts)
    else:
        from oracle import oracle as O
        O.VoxelGenerator(C2_BOUNDS, C2_SHAPE, **C2_KW)(pts)
    return time.perf_counter() - t0


def _cpu_iou_block(args):
    import torch
    torch.set_num_threads(1)
    seed, lo, hi = args
    rng = np.random.default_rng(seed)
    A, B = gen_boxes(rng, hi).astype(np.float32)[lo:hi], gen_boxes(rng, 4000).astype(np.float32)
    t0 = time.perf_counter()
    if _CPU_KIND == "reference":
        from oracle import ref as R
        R.box2d_iou(A, B, "rbox", precise=False)
    else:
        from oracle import oracle as O
        O.iou2dr(A, B)
    return time.perf_counter() - t0, (hi - lo) * 4000


def _cpu_iou64_block(args):
    import torch
    torch.set_num_threads(1)
    seed, lo, hi = args
    rng = np.random.default_rng(seed)
    A, B = gen_boxes(rng, hi)[lo:hi], gen_boxes(rng, 4000)
    t0 = time.perf_counter()
    if _CPU_KIND == "reference":
        from oracle import ref as R
        R.box2d_iou(A, B, "rbox", precise=True)
    else:
        from oracle import oracle as O
        O.iou2dr(A, B)
    return time.perf_counter() - t0, (hi - lo) * 4000


def _cpu_c5_frame(seed):
    """one C5 frame on the CPU: voxelize a C2 cloud, then rotated NMS of 4096 proposals"""
    import torch
    torch.set_num_threads(1)
    pts = lidar(500 + seed)
    P, s = proposals(900 + seed, 4096, 160)
    t0 = time.perf_counter()
    if _CPU_KIND == "reference":
        from oracle import ref as R
        R.VoxelGenerator(C2_BOUNDS, C2_SHAPE, **C2_KW)(pts)
        R.box2d_nms(P, s, "rbox", iou_threshold=0.5)
    else:
        from oracle import oracle as O
        O.VoxelGenerator(C2_BOUNDS, C2_SHAPE, **C2_KW)(pts)
        O.box2d_nms(P, s, "rbox", iou_threshold=0.5)
    return time.perf_counter() - t0


def gen_boxes3d(rng, n):
    b = gen_boxes(rng, n)
    return np.stack([b[:, 0], b[:, 1], rng.normal(-1.0, 0.5, n), b[:, 2], b[:, 3], 1.4 + rng.random(n) * 0.6, b[:, 4]], 1)


def _cpu_dist3d_block(args):
    import torch
    torch.set_num_threads(1)
    seed, lo, hi = args
    rng = np.random.default_rng(seed)
    A, B = gen_boxes3d(rng, hi).astype(np.float32)[lo:hi], gen_boxes3d(rng, 4000).astype(np.float32)
    from oracle import oracle as O
    t0 = time.perf_counter()
    O.box3d_iou_distance(A, B, "riou")
    return time.perf_counter() - t0, (hi - lo) * 4000


def _cpu_crop_block(args):
    import torch
    torch.set_num_threads(1)
    seed, nb = args
    rng = np.random.default_rng(seed)
    pts = lidar(seed, 180_000)[:, :2].copy()
    bx = proposals(seed, nb, max(1, nb // 2), extent=75.0)[0].astype(np.float32)
    t0 = time.perf_counter()
    if _CPU_KIND == "reference":
        from oracle import ref as R
        R.crop_2dr(pts, bx)
    else:
        from oracle import oracle as O
        O.crop_2dr(pts, bx)
    return time.perf_counter() - t0, len(pts) * nb


def c2s_inputs(seed=1):
    """SURVEY 8(d) C2s: the in-range points of a C2 cloud as (batch 0, x / 0.1, (y + 40) / 0.1) against f32[1,64,704,800]"""
    import torch
    pts = lidar(seed)
    ok = (pts[:, 0] >= 0) & (pts[:, 0] < 70.4) & (pts[:, 1] >= -40) & (pts[:, 1] < 40)
    p = pts[ok]
    coords = np.stack([np.zeros(len(p), np.float32), p[:, 0] / np.float32(0.1), (p[:, 1] + np.float32(40)) / np.float32(0.1)], 1).astype(np.float32)
    fmap = torch.rand((1, 64, 704, 800), generator=torch.Generator().manual_seed(7))
    return coords, fmap


def _cpu_scatter(method):
    import torch
    torch.set_num_threads(1)
    coords, fmap = c2s_inputs()
    t0 = time.perf_counter()
    if _CPU_KIND == "reference":
        from oracle import ref as R
        R.aligned_scatter_forward(coords, fmap.numpy(), method)
    else:
        from oracle import oracle as O
        O.scatter_forward(coords, fmap.numpy(), {"mean": 1, "linear": 2}[method])
    return time.perf_counter() - t0, len(coords)


def _cpu_nms(n):
    import torch
    torch.set_num_threads(1)
    P, s = proposals(2, n, max(1, n // 25))
    t0 = time.perf_counter()
    if _CPU_KIND == "reference":
        from oracle import ref as R
        R.box2d_nms(P, s, "rbox", iou_threshold=0.5)
    else:
        from oracle import oracle as O
        O.box2d_nms(P, s, "rbox", iou_threshold=0.5)
    return time.perf_counter() - t0


_CPU_KIND = "port"


def _cpu_child(fn, item, q):
    try:
        q.put((True, fn(item)))
    except BaseException as e:   # noqa: BLE001 -- report and carry on
        q.put((False, repr(e)))


def cpu_pool(fn, items, cores, timeout=240.0):
    """One forked process per work item, `cores` at a time (must run before CUDA is initialised in this
    process).  A multiprocessing.Pool would hang for ever when a worker dies, and the reference's fp32
    Rotating-Calipers path does die ("stack smashing detected": dgal's Poly2<T,8> vertex buffer overflows on
    some near-parallel pairs), so every item is isolated: a crashed or timed-out item yields None."""
    import multiprocessing as mp
    ctx = mp.get_context("fork")
    res = [None] * len(items)
    t0 = time.perf_counter()
    pending, running = list(enumerate(items)), []
    while pending or running:
        while pending and len(running) < cores:
            i, it = pending.pop(0)
            q = ctx.SimpleQueue()
            p = ctx.Process(target=_cpu_child, args=(fn, it, q))
            p.start()
            running.append((i, p, q))
        still = []
        for i, p, q in running:
            if not q.empty():
                ok, val = q.get()
                res[i] = val if ok else None
                p.join(5)
            elif not p.is_alive():
                p.join()
            elif time.perf_counter() - t0 > timeout:
                p.terminate(); p.join()
            else:
                still.append((i, p, q))
        running = still
        if running:
            time.sleep(0.002)
    return res, time.perf_counter() - t0


def cpu_baseline(op, cores, rounds=2):
    """Aggregate throughput of the reference CPU path with `rounds` units of work per host core (about
    10-30 s of CPU work in total).  Items that crash the reference are isolated, not counted, and reported."""
    global _CPU_KIND
    _CPU_KIND = _cpu_kind()
    if op == "voxel":
        res, wall = cpu_pool(_cpu_voxel_frame, [1000 + i for i in range(cores * rounds)], cores)
        ok = [r for r in res if r is not None]
        return dict(value=len(ok) * C2_POINTS / wall, unit="points/s", cores=cores, kind=_CPU_KIND,
                    sample=f"{len(ok)} C2 frames of {C2_POINTS} points, one frame per process on {cores} cores "
                           f"(single-frame latency {np.median(ok) * 1e3:.0f} ms, {len(res) - len(ok)} failed)")
    if op == "iou":
        rows = 256
        res, wall = cpu_pool(_cpu_iou_block, [(3, i * rows, (i + 1) * rows) for i in range(cores * rounds)], cores)
        ok = [r for r in res if r is not None]
        pairs = sum(r[1] for r in ok)
        return dict(value=pairs / wall, unit="pairs/s", cores=cores, kind=_CPU_KIND, crashed_blocks=len(res) - len(ok),
                    sample=f"{len(res)} row-blocks of {rows} x 4000 fp32 boxes (C4 distribution, precise=False), one block per "
                           f"process on {cores} cores; {len(res) - len(ok)} block(s) aborted inside the reference "
                           f"(dgal fp32 Rotating-Calipers overflows its Poly2<T,8> buffer: 'stack smashing detected') and are not counted")
    if op == "iou_f64":
        rows = 256
        res, wall = cpu_pool(_cpu_iou64_block, [(3, i * rows, (i + 1) * rows) for i in range(cores * rounds)], cores)
        ok = [r for r in res if r is not None]
        return dict(value=sum(r[1] for r in ok) / wall, unit="pairs/s", cores=cores, kind=_CPU_KIND, crashed_blocks=len(res) - len(ok),
                    sample=f"{len(res)} row-blocks of {rows} x 4000 fp64 boxes (C1 distribution, precise=True), one block per process on {cores} cores")
    if op == "c5":
        res, wall = cpu_pool(_cpu_c5_frame, list(range(cores * rounds)), cores)
        ok = [r for r in res if r is not None]
        return dict(value=len(ok) / wall, unit="frames/s", cores=cores, kind=_CPU_KIND,
                    sample=f"{len(ok)} C5 frames (C2 cloud + 4096 proposals), one frame per process on {cores} cores; single-frame latency {np.median(ok) * 1e3:.0f} ms")
    if op == "dist3d":
        rows = 256
        res, wall = cpu_pool(_cpu_dist3d_block, [(3, i * rows, (i + 1) * rows) for i in range(cores * rounds)], cores)
        ok = [r for r in res if r is not None]
        return dict(value=sum(r[1] for r in ok) / wall, unit="pairs/s", cores=cores, kind="port", crashed_blocks=len(res) - len(ok),
                    sample=f"{len(res)} row-blocks of {rows} x 4000 fp32 3-D boxes, one block per process on {cores} cores; C restatement of the "
                           f"reference's fp32 Rotating-Calipers IoU + the z arithmetic of d3d/dgal_wrap.h:45-68 (the reference's Cython matcher "
                           f"cannot be built in this image)")
    if op == "scatter":
        res, wall = cpu_pool(_cpu_scatter, ["linear"] * cores, cores)
        ok = [r for r in res if r is not None]
        return dict(value=sum(r[1] for r in ok) / wall, unit="points/s", cores=cores, kind=_CPU_KIND,
                    sample=f"{len(ok)} C2s forward passes (method linear, {ok[0][1] if ok else 0} points x 64 channels), one per process on {cores} cores; "
                           f"single-pass latency {np.median([r[0] for r in ok]) * 1e3:.0f} ms")
    if op == "crop":
        nb = 256
        res, wall = cpu_pool(_cpu_crop_block, [(200 + i, nb) for i in range(cores * rounds)], cores)
        ok = [r for r in res if r is not None]
        return dict(value=sum(r[1] for r in ok) / wall, unit="pairs/s", cores=cores, kind=_CPU_KIND,
                    sample=f"{len(ok)} blocks of {nb} boxes x 180000 points (fp32), one block per process on {cores} cores")
    if op == "nms":
        n = 10000
        res, wall = cpu_pool(_cpu_nms, [n] * (cores * rounds), cores)
        ok = [r for r in res if r is not None]
        return dict(value=len(ok) * n / wall, unit="boxes/s", cores=cores, kind=_CPU_KIND,
                    sample=f"{len(ok)} frames of {n} clustered proposals (C3 generator; the quadratic reference needs ~25 s for "
                           f"one 50k frame), one frame per process on {cores} cores; single-frame latency {np.median(ok) * 1e3:.0f} ms")
    raise ValueError(op)


# ------------------------------------------------------------------ clocks
class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thr = threading.Thread(target=self._read, daemon=True)
            self.thr.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def __exit__(self, *a):
        if self.proc:
            time.sleep(0.15)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def hold(self, fn, min_s=0.45):
        """the timed region of a short operator ends before nvidia-smi answers once: keep the same operator running (untimed)
        until the sampler has seen the GPU under this load"""
        import torch
        if not self.proc:
            return
        t0, n0 = time.time(), len(self.rows)
        while time.time() - t0 < min_s or (len(self.rows) < n0 + 2 and time.time() - t0 < 2.0):
            for _ in range(8):
                fn()
            torch.cuda.synchronize()

    def summary(self):
        sm, mx, reasons = [], 0.0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx = max(mx, float(r[1]))
                for nm, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                pass
        busy = [x for x in sm if x > 0.6 * mx] or sm
        return dict(sm_mhz=float(np.median(busy)) if busy else None, sm_max_mhz=mx or None, reasons=sorted(reasons), samples=len(sm))


# ------------------------------------------------------------------ GPU timing helpers
def timed(fn, steps, warmup, barrier, last=None):
    """ms per step of `steps` calls of fn after `warmup` untimed ones; `last` (a list) receives what the final timed call returned"""
    import torch
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        if last is not None and i == steps - 1:
            last.append(fn())
        else:
            fn()
    e1.record()
    torch.cuda.synchronize()
    barrier()
    return e0.elapsed_time(e1) / steps   # ms per step


def timed_flushed(fn, steps, warmup, barrier, last=None, before_last=None):
    """for operators whose working set fits L2: every step is timed by its own event pair and a 256 MB memset (outside the
    pairs) evicts L2 between steps; `last` as in timed(); `before_last` runs ahead of the final step's memset"""
    import torch
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    barrier()
    evs = []
    for i in range(steps):
        if before_last is not None and i == steps - 1:
            before_last()
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        if last is not None and i == steps - 1:
            last.append(fn())
        else:
            fn()
        e1.record()
        evs.append((e0, e1))
    torch.cuda.synchronize()
    barrier()
    return sum(a.elapsed_time(b) for a, b in evs) / steps


# ------------------------------------------------------------------ --dump-outputs
DUMP_SAMPLE = 1 << 18   # elements kept of one output array: at most 2 MB each, well under 64 MB for all operators together
DUMP_LIMIT = 64 << 20
OUTPUTS = {}            # name -> host array of the last timed step, written by main() when --dump-outputs is given


def keep_output(args, name, t):
    """Record what the timed path returned in its last step, as float32 (float32 and bool outputs) or float64 (float64 and integer
    outputs, exact).  An array of more than DUMP_SAMPLE elements is reduced to the elements at a fixed, seeded set of flat positions,
    so that two builds run with the same arguments can be compared output for output."""
    if not args.dump_outputs:
        return
    import torch
    flat = t.detach().reshape(-1)
    if flat.numel() > DUMP_SAMPLE:
        idx = np.unique(np.random.default_rng(0).integers(0, flat.numel(), DUMP_SAMPLE))
        a = flat[torch.from_numpy(idx).to(flat.device)].cpu().numpy()
    else:
        a = t.detach().cpu().numpy()
    OUTPUTS[name] = a.astype(np.float32 if a.dtype in (np.float32, np.bool_) else np.float64)


def keep_voxel_outputs(args, prefix, res):
    """the packed arrays of a VoxelBatch up to its totals: every frame's result dict is a slice of these"""
    if not args.dump_outputs:
        return
    rows = res.rows_host()
    K, V = int(rows[-1, 0]), int(rows[-1, 1])
    keep_output(args, f"{prefix}_rows", rows)
    for k, v in res.packed.items():
        keep_output(args, f"{prefix}_{k}", v[:K] if k in res.POINT_KEYS else v[:V])


def write_outputs(d):
    total = sum(a.nbytes for a in OUTPUTS.values())
    if total > DUMP_LIMIT:
        raise RuntimeError(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT}-byte limit")
    os.makedirs(d, exist_ok=True)
    for name, a in OUTPUTS.items():
        np.save(os.path.join(d, name + ".npy"), a)


def bind_to_gpu_numa(local):
    """Run this rank (and place the pinned staging memory it allocates afterwards: first touch) on the NUMA node of its GPU.  Without it
    every rank of a torchrun launch inherits the same affinity and all PCIe traffic of an 8-GPU box crosses one socket."""
    try:
        import torch
        pr = torch.cuda.get_device_properties(local)
        addr = f"{pr.pci_domain_id:04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
        node = int(open(f"/sys/bus/pci/devices/{addr}/numa_node").read())
        if node < 0:
            return dict(node=None, pci=addr)
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        allowed = os.sched_getaffinity(0)
        use = (cpus & allowed) or cpus
        os.sched_setaffinity(0, use)
        return dict(node=node, pci=addr, cpus=len(use))
    except Exception as e:   # affinity is an optimisation, never required
        return dict(node=None, error=repr(e)[:120])


def max_over_ranks(x, world):
    import torch
    if world == 1:
        return x
    import torch.distributed as dist
    t = torch.tensor([x], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def sum_over_ranks(x, world):
    import torch
    if world == 1:
        return x
    import torch.distributed as dist
    t = torch.tensor([x], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return float(t.item())


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def fma_peak(dtype_code):
    """measured CUDA-core FMA peak in TFLOP/s (FMA = 2 flops) with the library's probe kernel"""
    import ctypes as C
    import torch
    from d3d_b200 import _cabi as c
    sink = torch.zeros(4, device="cuda")
    fl = C.c_double(0)
    iters = 1 << 15 if dtype_code == 0 else 1 << 14
    best = 0.0
    for _ in range(4):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        c.check(c.fma_peak_probe(dtype_code, iters, c.ptr(sink), C.byref(fl), c.stream_ptr()), "fma probe")
        e1.record()
        torch.cuda.synchronize()
        best = max(best, fl.value / (e0.elapsed_time(e1) * 1e-3) / 1e12)
    return best


def ref_cuda_baseline(op):
    """Secondary GPU baseline: the reference's OWN CUDA kernels (d3d/box/iou_cuda.cu, nms_cuda.cu), compiled unmodified for sm_100a into
    oracle/_ref/box_impl_cuda (oracle/build_ref.py --cuda), on sizes their 32-bit pair index allows, next to this build on the same
    inputs.  Returns None when the module is not there."""
    import torch
    try:
        from oracle import build_ref
        m = build_ref.load_ref(build_ref.CUDA_MODULE)
    except Exception:
        return None
    from d3d_b200.box import box2d_iou, box2d_nms
    rng = np.random.default_rng(3)

    def ev(fn, reps=3):
        fn(); torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record(); torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps
    if op == "iou":
        # fp64, the reference's default dtype: its fp32 Rotating-Calipers path overruns a fixed-size vertex buffer on ~15 % of generic blocks
        # (CPU: "stack smashing detected"; GPU: illegal address).  The reference keeps u8[N, M, 8] flags for its backward and indexes pairs
        # with int32, so the square stays well below 16000.
        n = 8192
        A, B = torch.from_numpy(gen_boxes(rng, n)).cuda(), torch.from_numpy(gen_boxes(rng, n)).cuda()
        ms_ref = ev(lambda: m.iou2dr_forward_cuda(A, B), 2)
        ms_own = ev(lambda: box2d_iou(A, B, "rbox"))
        ref = m.iou2dr_forward_cuda(A[:2000], B[:2000])[0]
        own = box2d_iou(A[:2000], B[:2000], "rbox")
        return dict(workload=f"rotated IoU {n}x{n} fp64, C1 distribution", ref_cuda_ms=ms_ref, this_build_ms=ms_own, speedup=ms_ref / ms_own,
                    ref_cuda_pairs_per_s=n * n / (ms_ref * 1e-3), max_abs_diff_2000x2000=float((ref - own).abs().max()))
    if op == "nms":
        n = 20000
        P, sc = proposals(2, n, 800)
        tP, ts = torch.from_numpy(P).cuda(), torch.from_numpy(sc).cuda()
        it, st = m.IouType.RBOX, m.SupressionType.HARD
        ms_ref = ev(lambda: m.nms2d_cuda(tP, ts, it, st, 0.5, 0.0, 0.0), 2)
        ms_own = ev(lambda: box2d_nms(tP, ts, "rbox", iou_threshold=0.5))
        same = bool(torch.equal(~m.nms2d_cuda(tP, ts, it, st, 0.5, 0.0, 0.0), box2d_nms(tP, ts, "rbox", iou_threshold=0.5)))
        return dict(workload=f"rotated NMS {n} clustered proposals fp64, thr 0.5", ref_cuda_ms=ms_ref, this_build_ms=ms_own, speedup=ms_ref / ms_own,
                    ref_cuda_boxes_per_s=n / (ms_ref * 1e-3), same_keep_mask=same)
    return None


def alu_roofline(dtype_code, achieved_tflops, clocks):
    """roofline entry of an ALU-bound operator: against the measured FMA peak of this run (FFMA2 / DFMA probe), the nominal peak at the
    maximum clock and the nominal peak at the clock sampled under the operator's load"""
    lanes = 128 if dtype_code == 0 else 64
    peak = fma_peak(dtype_code)
    nominal = 148 * lanes * 2 * 1.965e9 / 1e12
    mhz = (clocks or {}).get("sm_mhz") or 1965.0
    at_clock = 148 * lanes * 2 * mhz * 1e6 / 1e12
    return dict(bound="fp32_alu" if dtype_code == 0 else "fp64_alu", achieved=achieved_tflops, peak=peak, unit="TFLOP/s", frac=achieved_tflops / peak, traffic=None,
                peak_source="measured in this run: d3d_fma_peak_probe, 16 chains/thread of " + ("FFMA2" if dtype_code == 0 else "DFMA"),
                peak_nominal=nominal, frac_nominal=achieved_tflops / nominal, peak_at_sampled_clock=at_clock, frac_at_sampled_clock=achieved_tflops / at_clock,
                probe_frac_of_nominal_at_sampled_clock=peak / at_clock)


# ------------------------------------------------------------------ operators
def bench_voxel(args, rank, world, barrier):
    import torch
    from d3d_b200 import _cabi as c
    from d3d_b200.voxel import VoxelGenerator
    F = args.frames
    frames = [lidar(100 + rank * F + i) for i in range(F)]      # weak scaling: every rank owns F distinct frames
    host = [torch.from_numpy(f).pin_memory() for f in frames]
    offs = torch.zeros(F + 1, dtype=torch.int64)
    offs[1:] = torch.tensor([len(f) for f in frames]).cumsum(0)
    dev_pts = torch.cat([h.cuda() for h in host], 0)
    gen = VoxelGenerator(C2_BOUNDS, C2_SHAPE, **C2_KW)
    offs_dev = offs.cuda()
    res = gen.batch_packed(dev_pts, offs, offs_dev)
    rows = res.rows_host()
    K, V = int(rows[-1, 0]), int(rows[-1, 1])
    N = int(dev_pts.shape[0])
    alg_bytes = 16.0 * N + 32.0 * K + 28.0 * V
    del res
    last = [] if args.dump_outputs else None
    l0 = c.launch_count()
    with ClockSampler(torch.cuda.current_device()) as cs:
        ms = timed(lambda: gen.batch_packed(dev_pts, offs, offs_dev), args.steps, args.warmup, barrier, last)
        l1 = c.launch_count()
        if last:
            keep_voxel_outputs(args, "voxel", last.pop())
        cs.hold(lambda: gen.batch_packed(dev_pts, offs, offs_dev))
    launches = (l1 - l0) // (args.steps + args.warmup) * args.steps
    ms = max_over_ranks(ms, world)
    e2e_steps = max(2, min(args.steps, 4))
    ms_e2e = max_over_ranks(timed(lambda: gen.batch(host), e2e_steps, 1, barrier), world)
    # one frame per call (the reference API): device-timed and end to end
    one_dev, one_offs = dev_pts[:C2_POINTS], offs[:2].clone()
    ms_one = max_over_ranks(timed(lambda: gen.batch_packed(one_dev, one_offs), max(args.steps, 20), 3, barrier), world)
    ms_one_e2e = max_over_ranks(timed(lambda: gen(host[0]), 10, 2, barrier), world)
    hbm, how = peaks()
    ach = alg_bytes / (ms * 1e-3) / 1e9
    traffic = None   # DRAM bytes per launch from the committed ncu capture, when it was taken on this workload
    try:
        with open(os.path.join(ROOT, "profiles", "r2_traffic.json")) as fh:
            t = json.load(fh)["voxel"]
        if t["frames"] == F and t["points_per_frame"] == C2_POINTS:
            traffic = float(t["bytes"])
    except (OSError, KeyError, ValueError):
        pass
    return dict(metric="voxelized points/sec", unit="points/s", value=N * world / (ms * 1e-3), ms_per_step=ms, dtype="f32",
                scaling="weak", gpu_launches=int(launches),
                config=dict(workload=f"C2 KITTI-shaped voxelization: {F} frames/GPU x {C2_POINTS} pts/frame, voxel 0.05x0.05x0.1 m "
                                     f"(grid 1408x1600x40), max 5 pts/voxel (trim), sparse VoxelGenerator path",
                            frames_per_gpu=F, points_per_frame=C2_POINTS, kept_points=K, voxels=V,
                            l2_policy=f"inputs larger than L2 ({N * 16 / 1e6:.0f} MB of points per step vs 126 MB L2)"),
                e2e=dict(value=N * world / (ms_e2e * 1e-3), unit="points/s", h2d_bytes_per_step=int(N * 16 + offs.numel() * 8),
                         d2h_bytes_per_step=int(16 * K + 28 * V + (F + 8) * 16), ms_per_step=ms_e2e,
                         api="VoxelGenerator.batch(list of pinned host tensors) -> host tensors (points = input[points_mask] is gathered on the host on first read)"),
                roofline=dict(bound="hbm", achieved=ach, peak=hbm, unit="GB/s", frac=ach / hbm, traffic=traffic, peak_source=how,
                              traffic_source="profiles/r2_traffic.json (ncu dram__bytes_read.sum + dram__bytes_write.sum summed over the step's four kernels)",
                              kernel="vt_split / vt_bucket / vt_scan / vt_write (voxel_tiles.cu): four launches per chunk of frames; algorithmic bytes 16N+32K+28V'",
                              algorithmic_bytes_per_step=alg_bytes),
                single_frame=dict(ms_device=ms_one, points_per_s=C2_POINTS / (ms_one * 1e-3), ms_e2e=ms_one_e2e, e2e_points_per_s=C2_POINTS / (ms_one_e2e * 1e-3),
                                  note="one 120k-point frame per call (the reference's call shape); bound by launch latency of the call's 7 launches"),
                clocks=cs.summary())


def bench_iou(args, rank, world, barrier, f64=False):
    import torch
    from d3d_b200 import _cabi as c
    from d3d_b200.box import box2d_iou, _pairwise
    from d3d_b200.parallel import row_block
    n = m = args.iou_f64_n if f64 else args.iou_n
    code, npdt, tdt, esz = (1, np.float64, torch.float64, 8) if f64 else (0, np.float32, torch.float32, 4)
    rng = np.random.default_rng(3)
    A, B = gen_boxes(rng, n).astype(npdt), gen_boxes(rng, m).astype(npdt)
    lo, hi = row_block(n, rank, world)                 # strong scaling: row-blocks of the same N x M matrix
    tA, tB = torch.from_numpy(A[lo:hi]).cuda(), torch.from_numpy(B).cuda()
    out = torch.empty((hi - lo, m), dtype=tdt, device="cuda")
    # candidate pairs of this rank's slab (roofline accounting only, outside the timed region)
    cnt = torch.zeros(64, dtype=torch.int64, device="cuda")
    ws = c.workspace(c.iou_workspace_bytes(hi - lo, m, code), tA.device)
    c.check(c.iou_count_candidates(c.ptr(tA), hi - lo, c.ptr(tB), m, code, c.ptr(cnt), c.ptr(ws), ws.numel(), c.stream_ptr()), "count")
    ncand = float(cnt.sum().item())
    pairs = float(hi - lo) * m
    l0 = c.launch_count()
    with ClockSampler(torch.cuda.current_device()) as cs:
        ms = timed(lambda: _pairwise(tA, tB, c.iou2dr, out), args.steps, args.warmup, barrier)
        l1 = c.launch_count()
        keep_output(args, "iou_f64" if f64 else "iou", out)
        cs.hold(lambda: _pairwise(tA, tB, c.iou2dr, out))
    launches = (l1 - l0) // (args.steps + args.warmup) * args.steps
    ms = max_over_ranks(ms, world)
    tot_pairs, tot_cand = sum_over_ranks(pairs, world), sum_over_ranks(ncand, world)
    flops = tot_cand * W_CAND + (tot_pairs - tot_cand) * W_REJ
    ach = flops / (ms * 1e-3) / 1e12 / world
    # e2e: host boxes in, a row-block slab of the matrix back on the host
    er = min(hi - lo, args.iou_e2e_rows)
    hA, hB = torch.from_numpy(A[lo:lo + er]).pin_memory(), torch.from_numpy(B).pin_memory()
    hout = torch.empty((er, m), dtype=tdt).pin_memory()

    def e2e_step():
        r = box2d_iou(hA.cuda(non_blocking=True), hB.cuda(non_blocking=True), "rbox", precise=f64)
        hout.copy_(r, non_blocking=True)
        torch.cuda.current_stream().synchronize()
    ms_e2e = max_over_ranks(timed(e2e_step, 3, 1, barrier), world)
    hbm, _ = peaks()
    clk = cs.summary()
    roof = alu_roofline(code, ach, clk)
    roof.update(algorithmic_flops=f"{W_CAND:.0f} per candidate pair + {W_REJ:.0f} per rejected pair (SURVEY.md 8(d): a candidate is a pair whose bounding circles "
                                  "overlap, counted by count_candidates_kernel; the tile kernel's own reject test passes fewer pairs to the clip)",
                store_gbs=tot_pairs * esz / (ms * 1e-3) / 1e9 / world, store_frac_of_hbm=tot_pairs * esz / (ms * 1e-3) / 1e9 / world / hbm)
    return dict(metric="rotated-IoU pairs/sec", unit="pairs/s", value=tot_pairs / (ms * 1e-3), ms_per_step=ms, dtype="f64" if f64 else "f32", scaling="strong",
                gpu_launches=int(launches),
                config=dict(workload=(f"rotated IoU {n}x{m} fp64 (precise=True), C1 distribution" if f64 else
                                      f"C4 detection-eval rotated IoU {n}x{m} fp32 (precise=False), C1 distribution") + f", row-block sharded over {world} GPU(s)",
                            candidate_fraction=tot_cand / tot_pairs,
                            l2_policy=f"output slab {pairs * esz / 1e9:.1f} GB per GPU streams through HBM, far larger than L2"),
                e2e=dict(value=er * m * world / (ms_e2e * 1e-3), unit="pairs/s", h2d_bytes_per_step=int((er + m) * 5 * esz),
                         d2h_bytes_per_step=int(er * m * esz), ms_per_step=ms_e2e,
                         api=f"box2d_iou(pinned host boxes [{er},5],[{m},5]) -> host [{er},{m}] slab"),
                roofline=roof, clocks=clk)


def bench_dist3d(args, rank, world, barrier):
    """SURVEY 8(f) f1: the detection evaluator's distance matrix 1 - iou2d * ziou over C4-sized 3-D box sets"""
    import torch
    from d3d_b200 import _cabi as c
    from d3d_b200.box import box3d_iou_distance
    from d3d_b200.parallel import row_block
    n = m = args.iou_n
    rng = np.random.default_rng(3)
    A, B = gen_boxes3d(rng, n).astype(np.float32), gen_boxes3d(rng, m).astype(np.float32)
    lo, hi = row_block(n, rank, world)
    tA, tB = torch.from_numpy(A[lo:hi]).cuda(), torch.from_numpy(B).cuda()
    out = torch.empty((hi - lo, m), dtype=torch.float32, device="cuda")
    bevA, bevB = tA[:, [0, 1, 3, 4, 6]].contiguous(), tB[:, [0, 1, 3, 4, 6]].contiguous()
    cnt = torch.zeros(64, dtype=torch.int64, device="cuda")
    ws = c.workspace(c.iou_workspace_bytes(hi - lo, m, 0), tA.device)
    c.check(c.iou_count_candidates(c.ptr(bevA), hi - lo, c.ptr(bevB), m, 0, c.ptr(cnt), c.ptr(ws), ws.numel(), c.stream_ptr()), "count")
    ncand, pairs = float(cnt.sum().item()), float(hi - lo) * m
    ws3 = c.workspace(c.iou3d_distance_workspace_bytes(hi - lo, m), tA.device)

    def step():
        c.check(c.iou3d_distance(c.ptr(tA), hi - lo, c.ptr(tB), m, 1, c.ptr(out), out.stride(0), c.ptr(ws3), ws3.numel(), c.stream_ptr()), "dist3d")
    l0 = c.launch_count()
    with ClockSampler(torch.cuda.current_device()) as cs:
        ms = timed(step, args.steps, args.warmup, barrier)
        l1 = c.launch_count()
        keep_output(args, "dist3d", out)
        cs.hold(step)
    launches = (l1 - l0) // (args.steps + args.warmup) * args.steps
    ms = max_over_ranks(ms, world)
    tot_pairs, tot_cand = sum_over_ranks(pairs, world), sum_over_ranks(ncand, world)
    peak32 = fma_peak(0)
    W_Z = 10.0   # z factor per CANDIDATE pair: 4 min/max, 2 subtractions, 2 clamps, divide, multiply, subtract (a rejected pair is the constant 1)
    flops = tot_cand * (W_CAND + W_Z) + (tot_pairs - tot_cand) * W_REJ
    ach = flops / (ms * 1e-3) / 1e12 / world
    er = min(hi - lo, args.iou_e2e_rows)
    hA, hB = torch.from_numpy(A[lo:lo + er]).pin_memory(), torch.from_numpy(B).pin_memory()
    hout = torch.empty((er, m), dtype=torch.float32).pin_memory()

    def e2e_step():
        r = box3d_iou_distance(hA.cuda(non_blocking=True), hB.cuda(non_blocking=True), "riou")
        hout.copy_(r, non_blocking=True)
        torch.cuda.current_stream().synchronize()
    ms_e2e = max_over_ranks(timed(e2e_step, 3, 1, barrier), world)
    hbm, _ = peaks()
    return dict(metric="evaluator distance-matrix pairs/sec", unit="pairs/s", value=tot_pairs / (ms * 1e-3), ms_per_step=ms, dtype="f32", scaling="strong",
                gpu_launches=int(launches),
                config=dict(workload=f"SURVEY 8(f) f1: ScoreMatcher distance cache 1 - riou2d * ziou, {n}x{m} fp32 3-D boxes (C4 BEV distribution), "
                                     f"row-block sharded over {world} GPU(s)", candidate_fraction=tot_cand / tot_pairs,
                            l2_policy=f"output slab {pairs * 4 / 1e9:.1f} GB per GPU streams through HBM, far larger than L2"),
                e2e=dict(value=er * m * world / (ms_e2e * 1e-3), unit="pairs/s", h2d_bytes_per_step=int((er + m) * 28),
                         d2h_bytes_per_step=int(er * m * 4), ms_per_step=ms_e2e,
                         api=f"box3d_iou_distance(pinned host boxes [{er},7],[{m},7]) -> host [{er},{m}] slab"),
                roofline=dict(bound="fp32_alu", achieved=ach, peak=peak32, unit="TFLOP/s", frac=ach / peak32, traffic=None,
                              peak_source="measured with d3d_fma_peak_probe in this run",
                              algorithmic_flops=f"{W_CAND:.0f} + {W_Z:.0f} (z factor) per candidate pair + {W_REJ:.0f} per rejected pair",
                              store_gbs=tot_pairs * 4 / (ms * 1e-3) / 1e9 / world),
                clocks=cs.summary())


def bench_crop(args, rank, world, barrier):
    """SURVEY 8(f) f4: point-in-rotated-box mask, one C3-sized frame (180k points) against 4096 boxes per GPU per step"""
    import torch
    from d3d_b200 import _cabi as c
    from d3d_b200.box import box2dr_crop
    n, m = 180_000 // 16 * 16, 4096
    pts = torch.from_numpy(lidar(300 + rank, 180_000)[:n, :2].copy()).cuda()
    bx = torch.from_numpy(proposals(300 + rank, m, m // 2)[0].astype(np.float32)).cuda()
    mask = torch.empty((m, n), dtype=torch.bool, device="cuda")
    ws = c.workspace(c.crop_workspace_bytes(n, m, 0), pts.device)

    def step():
        c.check(c.crop2dr[0](c.ptr(pts), n, c.ptr(bx), m, c.ptr(mask), c.ptr(ws), ws.numel(), c.stream_ptr()), "crop")
    l0 = c.launch_count()
    with ClockSampler(torch.cuda.current_device()) as cs:
        ms = timed(step, args.steps, args.warmup, barrier)
        l1 = c.launch_count()
        keep_output(args, "crop_mask", mask)
        cs.hold(step)
    launches = (l1 - l0) // (args.steps + args.warmup) * args.steps
    ms = max_over_ranks(ms, world)
    hP, hB = pts.cpu().pin_memory(), bx.cpu().pin_memory()
    hout = torch.empty((m, n), dtype=torch.bool).pin_memory()

    def e2e_step():
        r = box2dr_crop(hP.cuda(non_blocking=True), hB.cuda(non_blocking=True))
        hout.copy_(r, non_blocking=True)
        torch.cuda.current_stream().synchronize()
    ms_e2e = max_over_ranks(timed(e2e_step, 3, 1, barrier), world)
    hbm, how = peaks()
    alg = float(m) * n + 8.0 * n + 20.0 * m
    ach = alg / (ms * 1e-3) / 1e9
    return dict(metric="point-in-box pairs/sec", unit="pairs/s", value=float(m) * n * world / (ms * 1e-3), ms_per_step=ms, dtype="f32", scaling="weak",
                gpu_launches=int(launches),
                config=dict(workload=f"SURVEY 8(f) f4: box2dr_crop, {n} points x {m} rotated boxes fp32, one frame per GPU per step",
                            l2_policy=f"the {m * n / 1e6:.0f} MB mask streams through HBM, larger than L2"),
                e2e=dict(value=float(m) * n * world / (ms_e2e * 1e-3), unit="pairs/s", h2d_bytes_per_step=int(8 * n + 20 * m), d2h_bytes_per_step=int(m * n),
                         ms_per_step=ms_e2e, api="box2dr_crop(pinned host points, boxes) -> host bool mask"),
                roofline=dict(bound="hbm", achieved=ach, peak=hbm, unit="GB/s", frac=ach / hbm, traffic=None, peak_source=how,
                              algorithmic_bytes_per_step=alg, note="1 mask byte per pair, written once: a pure store stream zero-fills the mask (7 TB/s, tools/write_bw_probe.cu) "
                                                                    "while the points are binned into a grid on a high-priority internal stream; the hit kernels then set the few "
                                                                    "bytes of the candidates inside their box (brute force: D3D_B200_CROP_PATH=brute)"),
                clocks=cs.summary())


def bench_scatter(args, rank, world, barrier):
    """SURVEY 8(d) C2s: aligned_scatter forward + backward (method linear) of one C2 frame's points on a 64-channel BEV map"""
    import torch
    from d3d_b200 import _cabi as c
    from d3d_b200.point import aligned_scatter, aligned_scatter_forward_cuda, aligned_scatter_backward_cuda, AlignType
    coords_np, fmap = c2s_inputs(1 + rank)
    coords, fm = torch.from_numpy(coords_np).cuda(), fmap.cuda()
    n, ch = coords.shape[0], fm.shape[1]
    grad = torch.ones((n, ch), dtype=torch.float32, device="cuda")
    image_grad = torch.zeros_like(fm)

    from d3d_b200.point import ScatterPlan, _dims

    def fwd(plan=None):
        return aligned_scatter_forward_cuda(coords, fm, AlignType.LINEAR, plan)

    def step():
        plan = ScatterPlan(n, 2, fm.shape[0], _dims(fm.shape), fm.device)   # what AlignedScatter does: the backward reuses the forward's binning
        out = fwd(plan)
        aligned_scatter_backward_cuda(coords, grad, AlignType.LINEAR, image_grad, plan)   # accumulates in place (the caller zeroes once, d3d/point/__init__.py:32)
        return out
    anchor = float(fwd().double().sum().item())
    last = [] if args.dump_outputs else None
    l0 = c.launch_count()
    with ClockSampler(torch.cuda.current_device()) as cs:
        # when dumping, the map gradient is zeroed ahead of the last step (before its L2 flush) so that it holds that step's backward alone;
        # the backward reduce-adds into the map, so it is equal from run to run up to fp32 rounding
        ms = timed_flushed(step, args.steps, args.warmup, barrier, last, image_grad.zero_ if args.dump_outputs else None)
        l1 = c.launch_count()
        if last:
            keep_output(args, "scatter_forward", last.pop())
            keep_output(args, "scatter_image_grad", image_grad)
        ms_fwd = timed_flushed(fwd, args.steps, 1, barrier)
        cs.hold(step)
    launches = (l1 - l0) // (args.steps + args.warmup) * args.steps
    ms, ms_fwd = max_over_ranks(ms, world), max_over_ranks(ms_fwd, world)
    hC = torch.from_numpy(coords_np).pin_memory()

    def e2e_step():
        r = aligned_scatter(hC.cuda(non_blocking=True), fm, "linear")   # the feature map is an activation that already lives on the device
        r.cpu()
    ms_e2e = max_over_ranks(timed(e2e_step, 3, 1, barrier), world)
    hbm, how = peaks()
    dim = 2
    alg_f = n * ch * (2 ** dim + 1) * 4.0 + n * (1 + dim) * 4.0          # SURVEY 8(d): gather 2^Dim neighbours + write, per channel
    alg = 2 * alg_f                                                      # backward: read grad, read-modify-write 2^Dim neighbours
    ach = alg / (ms * 1e-3) / 1e9
    traffic = None
    try:
        with open(os.path.join(ROOT, "profiles", "r2_traffic.json")) as fh:
            t = json.load(fh)["scatter"]
        if t["points"] == n:
            traffic = float(t["bytes"])
    except (OSError, KeyError, ValueError):
        pass
    return dict(metric="aligned_scatter points/sec (forward + backward)", unit="points/s", value=n * world / (ms * 1e-3), ms_per_step=ms, dtype="f32",
                scaling="weak", gpu_launches=int(launches),
                config=dict(workload=f"SURVEY 8(d) C2s: {n} in-range points of a C2 frame, feature map f32[1,64,704,800], method linear, "
                                     f"forward + backward per step, one frame per GPU", forward_ms=ms_fwd, forward_sum_anchor=anchor,
                            l2_policy="256 MB memset evicts L2 between timed steps (the 144 MB map itself exceeds L2)"),
                e2e=dict(value=n * world / (ms_e2e * 1e-3), unit="points/s", h2d_bytes_per_step=int(n * 12), d2h_bytes_per_step=int(n * ch * 4),
                         ms_per_step=ms_e2e, api="aligned_scatter(pinned host coordinates, device feature map, 'linear') -> host [N,64]"),
                roofline=dict(bound="hbm", achieved=ach, peak=hbm, unit="GB/s", frac=ach / hbm, traffic=traffic, peak_source=how,
                              algorithmic_bytes_per_step=alg, forward_gbs=alg_f / (ms_fwd * 1e-3) / 1e9,
                              note="N*C*(2^Dim+1)*4 + N*(1+Dim)*4 bytes per pass (SURVEY 8(d)).  Tile path (scatter.cu): the points are binned by 8x64-cell tile, "
                                   "every tile is staged once in shared memory by a 3-D TMA tensor copy and the backward sends it back with a TMA reduce-add; "
                                   "DRAM traffic per pass = the 144 MB map + halo (ncu: forward 146 MB read + 13 MB written; profiles/r2_scatter_launches.txt). "
                                   "The gather path (D3D_B200_SCATTER_PATH=gather) pays a 32-byte sector per 4-byte neighbour: 352 MB forward, 0.31 ms per step"),
                clocks=cs.summary())


def bench_nms(args, rank, world, barrier):
    import torch
    from d3d_b200 import _cabi as c
    from d3d_b200.box import box2d_nms
    n = args.nms_n
    P, s = proposals(2 + rank, n)                      # weak scaling: one C3 frame per rank per step
    tP, ts = torch.from_numpy(P).cuda(), torch.from_numpy(s).cuda()
    keep = box2d_nms(tP, ts, "rbox", iou_threshold=0.5)
    kept = int(keep.sum().item())
    last = [] if args.dump_outputs else None
    l0 = c.launch_count()
    with ClockSampler(torch.cuda.current_device()) as cs:
        ms = timed_flushed(lambda: box2d_nms(tP, ts, "rbox", iou_threshold=0.5), args.steps, args.warmup, barrier, last)
        l1 = c.launch_count()
        if last:
            keep_output(args, "nms_keep", last.pop())
        cs.hold(lambda: box2d_nms(tP, ts, "rbox", iou_threshold=0.5))
    launches = (l1 - l0) // (args.steps + args.warmup) * args.steps
    ms = max_over_ranks(ms, world)
    hP, hs = torch.from_numpy(P).pin_memory(), torch.from_numpy(s).pin_memory()
    ms_e2e = max_over_ranks(timed(lambda: box2d_nms(hP, hs, "rbox", iou_threshold=0.5), 3, 1, barrier), world)
    # phase times: the same call truncated after sort + gather (knob 1) and after the candidate phase (knob 2)
    phase = {}
    for knob in (1, 2):
        c.tuning_set("D3D_B200_NMS_STOP", knob)
        phase[knob] = timed_flushed(lambda: box2d_nms(tP, ts, "rbox", iou_threshold=0.5), max(3, args.steps // 2), 2, barrier)
    c.tuning_set("D3D_B200_NMS_STOP", None)
    ms_sort, ms_pairs, ms_resolve = phase[1], max(phase[2] - phase[1], 1e-6), max(ms - phase[2], 1e-6)
    # clips of the candidate phase: pairs i < j in score order whose bounding circles overlap
    cnt = torch.zeros(64, dtype=torch.int64, device="cuda")
    ws = c.workspace(c.iou_workspace_bytes(n, n, 1), tP.device)
    c.check(c.iou_count_candidates(c.ptr(tP), n, c.ptr(tP), n, 1, c.ptr(cnt), c.ptr(ws), ws.numel(), c.stream_ptr()), "count")
    clips = max((float(cnt.sum().item()) - n) / 2.0, 0.0)
    clk = cs.summary()
    # soft-NMS (gaussian) of the reference's default shape: sequential in the kept boxes, a latency path; reported, not a roofline line
    soft = {}
    if rank == 0:
        for m in (1000, 4096):
            sP, ss = tP[:m].contiguous(), ts[:m].contiguous()
            f = lambda: box2d_nms(sP, ss, "rbox", "gaussian", iou_threshold=0.3, score_threshold=0.2, supression_param=0.5)  # noqa: E731
            soft[str(m)] = dict(ms=timed(f, 3, 1, lambda: None), kept=int(f().sum().item()))
    roof = alu_roofline(1, clips * W_CAND / (ms_pairs * 1e-3) / 1e12, clk)
    roof.update(phase="candidate phase (nms_cells_kernel): pairs whose bounding circles meet x 230 flop (SURVEY.md 8(d): the work a clip-every-candidate kernel "
                      "would do) over its own time; the kernel drops most of these pairs with an area bound before the clip, so its FP64 pipe is far less busy "
                      "than this fraction suggests (ncu: 7 %) -- read it as candidates per second, not as pipe utilisation", clips=clips, ms_sort_gather=ms_sort, ms_candidates=ms_pairs,
                ms_resolve=ms_resolve, resolve_us_per_64_box_block=ms_resolve * 1e3 / ((n + 63) // 64),
                note="the resolve is the fixpoint of keep / suppress decisions, pulled by a thread per box over the transposed hit lists (latency of the longest chain "
                     "of decisions: no roofline; D3D_B200_NMS_FIX=2: the same fixpoint by rounds with grid barriers, 0.23 ms; =0: the block-by-block walk in score order on one SM, 0.97 ms)")
    return dict(metric="NMS boxes/sec", unit="boxes/s", value=n * world / (ms * 1e-3), ms_per_step=ms, dtype="f64", scaling="weak",
                gpu_launches=int(launches),
                config=dict(workload=f"C3 BEV rotated NMS: {n} clustered proposals/frame (2000 objects), rbox thr 0.5, precise=True (fp64), "
                                     f"one frame per GPU per step", kept=kept,
                            l2_policy="working set (3 MB of box records, ~10 MB of suppression lists) fits L2: a 256 MB memset evicts L2 between "
                                      "timed steps, each step timed by its own event pair"),
                e2e=dict(value=n * world / (ms_e2e * 1e-3), unit="boxes/s", h2d_bytes_per_step=int(n * 48), d2h_bytes_per_step=int(n),
                         ms_per_step=ms_e2e, api="box2d_nms(pinned host boxes, scores) -> host keep mask"),
                roofline=roof, clocks=clk, soft=soft)


def bench_c5(args, rank, world, barrier):
    """BASELINE.json config 5: a batch of 64 frames, each a C2 cloud + 4096 BEV proposals, voxelize -> NMS, frames sharded over the GPUs
    (strong scaling), keep masks and voxel counts gathered over NCCL at the end; the gather is timed separately"""
    import torch
    from d3d_b200 import _cabi as c
    from d3d_b200.voxel import VoxelGenerator
    from d3d_b200.box import box2d_nms_batch
    from d3d_b200.parallel import frame_shard, gather_frames
    F, NP = args.c5_frames, 4096
    mine = frame_shard(F, rank, world)
    clouds = [lidar(500 + f) for f in mine]
    props = [proposals(900 + f, NP, 160) for f in mine]
    nf = len(mine)
    dev_pts = torch.cat([torch.from_numpy(x) for x in clouds], 0).cuda() if nf else torch.zeros((0, 4), device="cuda")
    offs = torch.zeros(nf + 1, dtype=torch.int64)
    offs[1:] = torch.tensor([len(x) for x in clouds], dtype=torch.int64).cumsum(0) if nf else 0
    offs_dev = offs.cuda()
    pb = torch.cat([torch.from_numpy(b) for b, _ in props], 0).cuda() if nf else torch.zeros((0, 5), dtype=torch.float64, device="cuda")
    ps = torch.cat([torch.from_numpy(s_) for _, s_ in props], 0).cuda() if nf else torch.zeros(0, dtype=torch.float64, device="cuda")
    poffs = torch.arange(nf + 1, dtype=torch.int64) * NP
    poffs_dev = poffs.cuda()
    gen = VoxelGenerator(C2_BOUNDS, C2_SHAPE, **C2_KW)
    state = {}

    def step():
        if nf:
            state["vox"] = gen.batch_packed(dev_pts, offs, offs_dev)
            state["keep"] = box2d_nms_batch(pb, ps, poffs, iou_method="rbox", iou_threshold=0.5, offsets_dev=poffs_dev)
    l0 = c.launch_count()
    with ClockSampler(torch.cuda.current_device()) as cs:
        ms = timed(step, args.steps, args.warmup, barrier)
        l1 = c.launch_count()
        if nf:
            keep_voxel_outputs(args, "c5_voxel", state["vox"])
            keep_output(args, "c5_keep", state["keep"])
        cs.hold(step)
    launches = (l1 - l0) // (args.steps + args.warmup) * args.steps
    ms = max_over_ranks(ms, world)

    def gather():
        keeps = [state["keep"][k * NP:(k + 1) * NP] for k in range(nf)]
        rows = state["vox"].rows if nf else torch.zeros((1, 2), dtype=torch.int64, device="cuda")
        nvox = [(rows[k + 1, 1] - rows[k, 1]).reshape(1) for k in range(nf)]
        gk = gather_frames(keeps, F, dtype=torch.bool, device=torch.device("cuda", torch.cuda.current_device()))
        gv = gather_frames(nvox, F, dtype=torch.int64, device=torch.device("cuda", torch.cuda.current_device()))
        return gk, gv
    step()
    ms_gather = max_over_ranks(timed(gather, 3, 1, barrier), world)
    gk, gv = gather()
    kept = int(sum(int(k.sum()) for k in gk))
    voxels = int(sum(int(v.item()) for v in gv))
    # end to end: pinned host clouds and proposals in, host keep masks and per-frame voxel results out
    hclouds = [torch.from_numpy(x).pin_memory() for x in clouds]
    hb = [torch.from_numpy(b).pin_memory() for b, _ in props]
    hs = [torch.from_numpy(s_).pin_memory() for _, s_ in props]

    def e2e_step():
        if nf:
            gen.batch(hclouds)
            box2d_nms_batch(hb, hs, iou_method="rbox", iou_threshold=0.5)
    ms_e2e = max_over_ranks(timed(e2e_step, 2, 1, barrier), world)
    weak = None
    if world > 1:
        # the same pipeline with the whole 64-frame batch on EVERY rank (weak scaling): what the box delivers when every GPU has a full batch,
        # beside the strong-scaling line above, whose per-rank share (F / world frames) is bound by the latency of the kernel chain
        wc = [lidar(500 + rank * F + f) for f in range(F)]
        wp = [proposals(900 + rank * F + f, NP, 160) for f in range(F)]
        w_pts = torch.cat([torch.from_numpy(x) for x in wc], 0).cuda()
        w_offs = torch.zeros(F + 1, dtype=torch.int64); w_offs[1:] = torch.tensor([len(x) for x in wc], dtype=torch.int64).cumsum(0)
        w_offs_dev = w_offs.cuda()
        w_pb = torch.cat([torch.from_numpy(b) for b, _ in wp], 0).cuda(); w_ps = torch.cat([torch.from_numpy(s_) for _, s_ in wp], 0).cuda()
        w_poffs = torch.arange(F + 1, dtype=torch.int64) * NP; w_poffs_dev = w_poffs.cuda()

        def wstep():
            gen.batch_packed(w_pts, w_offs, w_offs_dev)
            box2d_nms_batch(w_pb, w_ps, w_poffs, iou_method="rbox", iou_threshold=0.5, offsets_dev=w_poffs_dev)
        wms = max_over_ranks(timed(wstep, args.steps, args.warmup, barrier), world)
        weak = dict(frames_per_gpu=F, ms_per_step=wms, value=F * world / (wms * 1e-3), unit="frames/s", scaling="weak")
    return dict(metric="voxelize->NMS pipeline frames/sec", unit="frames/s", value=F / (ms * 1e-3), ms_per_step=ms, dtype="f32 voxels, f64 NMS", scaling="strong", weak=weak,
                gpu_launches=int(launches),
                config=dict(workload=f"C5: batch of {F} frames x (C2 cloud of {C2_POINTS} points + {NP} BEV proposals), voxelize -> rotated NMS thr 0.5, "
                                     f"frames sharded over {world} GPU(s)", frames=F, frames_this_rank=nf, kept_boxes=kept, voxels=voxels,
                            l2_policy=f"{nf * C2_POINTS * 16 / 1e6:.0f} MB of points per step on this rank"),
                e2e=dict(value=F / (ms_e2e * 1e-3), unit="frames/s", h2d_bytes_per_step=int(nf * (C2_POINTS * 16 + NP * 48)),
                         d2h_bytes_per_step=int(nf * NP + voxels / max(world, 1) * 28), ms_per_step=ms_e2e,
                         api="VoxelGenerator.batch(pinned host clouds) + box2d_nms_batch(pinned host boxes, scores) -> host results"),
                gather=dict(ms=ms_gather, what=f"keep masks ({F} x {NP} bool) + voxel counts of all frames, gather_frames over " + ("NCCL" if world > 1 else "one rank (no collective)")),
                roofline=dict(bound="hbm", achieved=None, peak=None, unit="GB/s", frac=None, traffic=None,
                              note="pipeline of the voxel and NMS operators; their rooflines are the top-level line and ops.nms"),
                clocks=cs.summary())


# ------------------------------------------------------------------ reference arm
def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    op = "voxel" if args.op == "all" else args.op
    vals = []
    for _ in range(args.warmup + args.steps):
        vals.append(cpu_baseline(op, cores))
    vals = vals[args.warmup:] or vals
    v = float(np.median([x["value"] for x in vals]))
    cb = dict(vals[-1]); cb["value"] = v
    metric = {"voxel": "voxelized points/sec", "iou": "rotated-IoU pairs/sec", "iou_f64": "rotated-IoU pairs/sec", "c5": "voxelize->NMS pipeline frames/sec", "nms": "NMS boxes/sec", "dist3d": "evaluator distance-matrix pairs/sec", "crop": "point-in-box pairs/sec", "scatter": "aligned_scatter points/sec (forward)"}[op]
    unit = cb["unit"]
    line = dict(impl="reference", metric=metric, value=v, unit=unit, n_gpus=args.gpus, steps=args.steps, warmup=args.warmup,
                ms_per_step=None, higher_is_better=True, scaling="weak", vs_baseline=None,
                dtype={"voxel": "f32", "iou": "f32", "iou_f64": "f64", "c5": "f32 voxels, f64 NMS", "nms": "f64", "dist3d": "f32", "crop": "f32", "scatter": "f32"}[op], data="synthetic",
                config=dict(workload={"voxel": "C2 KITTI-shaped voxelization 120k pts/frame, 0.05x0.05x0.1 m voxels, max 5 pts/voxel (reference CPU path)",
                                      "iou": "C4 rotated IoU fp32, C1 distribution (reference CPU path, row-block sample)",
                                      "iou_f64": "rotated IoU fp64, C1 distribution (reference CPU path, row-block sample)",
                                      "c5": "C5 frames: C2 cloud voxelization + rotated NMS of 4096 proposals (reference CPU path)",
                                      "nms": "C3-style rotated NMS fp64, 5000-proposal frames (reference CPU path)",
                                      "scatter": "C2s aligned_scatter forward, method linear (reference CPU path)",
                                      "crop": "box2dr_crop 180k points x 256-box blocks fp32 (reference CPU path)",
                                      "dist3d": "evaluator distance matrix 1 - riou2d * ziou fp32 (C restatement of the reference path, row-block sample)"}[op]),
                cpu_baseline=cb, e2e=dict(value=v, unit=unit, h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0)
    print(json.dumps(line))


# ------------------------------------------------------------------ main
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--op", default="all", choices=["all", "voxel", "iou", "iou_f64", "nms", "c5", "scatter", "dist3d", "crop"])
    ap.add_argument("--iou-f64-n", type=int, default=30_000)
    ap.add_argument("--c5-frames", type=int, default=64)
    ap.add_argument("--frames", type=int, default=128, help="C2 frames per GPU per voxelization step")
    ap.add_argument("--iou-n", type=int, default=100_000)
    ap.add_argument("--iou-e2e-rows", type=int, default=8192)
    ap.add_argument("--nms-n", type=int, default=50_000)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one computed as DIR/<name>.npy "
                                                          "(float32 or float64; larger outputs as a fixed, seeded sample; rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.impl == "reference":
        return run_reference(args)

    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        args.dump_outputs = None
    local = int(os.environ.get("LOCAL_RANK", "0"))
    ops = ["voxel", "iou", "nms", "iou_f64", "c5", "scatter", "dist3d", "crop"] if args.op == "all" else [args.op]

    # CPU baseline first: the fork-based pool must run before this process touches CUDA
    cpu = {}
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cores = os.cpu_count() or 1
        for op in ops:
            try:
                cpu[op] = cpu_baseline(op, cores)
            except Exception as e:   # the baseline is reported, never required
                cpu[op] = dict(value=None, unit=None, cores=cores, kind="unavailable", sample=str(e))

    import torch
    torch.cuda.set_device(local)
    numa = bind_to_gpu_numa(local)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        barrier = lambda: dist.barrier()
    else:
        barrier = lambda: None
    import d3d_b200  # noqa: F401  (raises if the CUDA extension is missing: no fallback)

    fns = dict(voxel=bench_voxel, iou=bench_iou, iou_f64=lambda *a: bench_iou(*a, f64=True), nms=bench_nms, c5=bench_c5, dist3d=bench_dist3d, crop=bench_crop,
               scatter=bench_scatter)
    res = {}
    for op in ops:
        res[op] = fns[op](args, rank, world, barrier)
        if op in cpu:
            res[op]["cpu_baseline"] = cpu[op]
        if world == 1 and op in ("iou", "nms") and not args.no_cpu_baseline:
            try:
                # in its own interpreter: the module registers the same pybind11 enums as the CPU build of the reference that the CPU arm loaded
                out = subprocess.run([sys.executable, "-c", f"import json, bench; print('REFCUDA', json.dumps(bench.ref_cuda_baseline({op!r})))"],
                                     cwd=ROOT, capture_output=True, text=True, timeout=600)
                got = [ln for ln in out.stdout.splitlines() if ln.startswith("REFCUDA ")]
                rc = json.loads(got[-1][8:]) if got else dict(unavailable=(out.stderr or out.stdout)[-200:])
            except Exception as e:   # a baseline, never required
                rc = dict(unavailable=repr(e)[:200])
            if rc:
                res[op]["ref_cuda"] = rc
        torch.cuda.empty_cache()
    if world > 1:
        # the only collective of the pipeline: small per-rank results are gathered at the end (outside the timed regions)
        from d3d_b200.parallel import gather_ragged
        gather_ragged(torch.tensor([res[ops[0]]["ms_per_step"]], device="cuda"))
        dist.barrier()
    if rank == 0:
        top = dict(res[ops[0]])
        line = dict(metric=top.pop("metric"), value=top.pop("value"), unit=top.pop("unit"), n_gpus=world, steps=args.steps, warmup=args.warmup,
                    ms_per_step=top.pop("ms_per_step"), higher_is_better=True, scaling=top.pop("scaling"), vs_baseline=None,
                    dtype=top.pop("dtype"), data="synthetic (seeded generators of SURVEY.md 8(d))")
        line.update(top)
        line.setdefault("cpu_baseline", None)
        line["numa"] = numa
        # the three north_star metrics as top-level keys (the other operators keep their full records under "ops")
        for op, keys in (("iou", ("iou_pairs_per_s", "iou_frac_of_fp32_peak")), ("nms", ("nms_boxes_per_s", "nms_candidate_frac_of_fp64_peak")),
                         ("iou_f64", ("iou_f64_pairs_per_s", "iou_f64_frac_of_fp64_peak")), ("c5", ("c5_frames_per_s", None))):
            if op in res:
                line[keys[0]] = res[op]["value"]
                if keys[1]:
                    line[keys[1]] = res[op]["roofline"].get("frac")
        if "c5" in res and res["c5"].get("weak"):   # config 5 with a full batch on every rank, beside the strong-scaling number
            line["c5_weak_frames_per_s"] = res["c5"]["weak"]["value"]
        if len(ops) > 1:
            line["ops"] = {op: res[op] for op in ops[1:]}
        if args.dump_outputs:
            write_outputs(args.dump_outputs)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
