#!/usr/bin/env python
"""bench.py — CSR SpMM throughput on B200 (BASELINE.json: "SpMM GFLOP/s & HBM GB/s (% roofline)
at K=32/256, 1/2/4/8 B200 vs host CPU").

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload reddit_k256] [--impl reference] [--dump-outputs DIR]

A step is one SpMM (C = A·B) of the named synthetic graph: every kernel `spmm_b200_run`
launches, through the C ABI. For N > 1 (torchrun) A's rows are partitioned by nnz over the ranks
(B replicated, no data-path collective), the timed region is bracketed by a barrier and a device
synchronise, the per-rank device time is taken with CUDA events and the MAX over ranks is
reported; `value` is the whole job's GFLOP/s = 2·nnz·K / step time ("strong" scaling: the graph
is fixed, each rank gets 1/N of its nonzeros).

`e2e` is the same step through the host-buffer call: N = 1 `spmm_b200_run_host` (B in over PCIe, C out);
N > 1 `spmm_b200_run_host_sharded` — every rank uploads only its 1/N slice of B and the ranks replicate it
over NVLink (multimem.st / peer stores), every rank downloads its own block of C.

With N > 1 the line also carries, under `also`, BASELINE config 5: the products-shaped graph over the same
ranks (SpMM alone, strong scaling) and two stacked layers with the all-gather of C done by NCCL (all-gather-v)
and by the kernel's own epilogue (peer / multicast stores), bit-compared.

`--dump-outputs DIR` (GPU arm only) writes C as the last timed step left it to DIR/C.npy, with its row numbers in
DIR/C_rows.npy; above DUMP_BYTES a fixed, seeded sample of rows (see dump_outputs).

`--impl reference` times the CPU restatement of the reference's SpMM (oracle/spmm_oracle.c,
OpenMP over rows — the reference itself has no CPU path: PA4/handout/src/spmm_ref.cu is a CUDA
kernel) on the box's host cores, on a bounded row sample of the same workload. That arm loads only
the host-side graph generator (hpc_b200/libspmm_b200_graph.so) and the oracle — no product kernel.
"""
from __future__ import annotations

import argparse
import ctypes
import hashlib
import importlib.util
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (graph shape, K)
    "c0_k32": ("c0", 32),
    "arxiv_k32": ("arxiv", 32),
    "arxiv_k256": ("arxiv", 256),
    "reddit_k32": ("reddit", 32),
    "reddit_k256": ("reddit", 256),
    "products_k256": ("products", 256),
}
SEED = 123
L2_BYTES = 126 << 20
NVLINK_PEER_GBS = 770.0   # measured peer copy per direction (B200_PROFILING.md)
DUMP_BYTES = 48 << 20     # --dump-outputs writes at most this much (C, or a seeded sample of its rows)


def bytes_min(m, nnz, k, b_rows=None):
    """SURVEY.md §8d: ptr + idx + val + B read once + C written once."""
    b_rows = m if b_rows is None else b_rows
    return 4 * (m + 1) + 8 * nnz + 4 * b_rows * k + 4 * m * k


def bytes_gather(m, nnz, k):
    return 4 * (m + 1) + 8 * nnz + 4 * nnz * k + 4 * m * k


def measured_peaks():
    try:
        d = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def workload_config(workload, ptr):
    """The `config` object — identical in both arms (same keys, same values) for the same workload."""
    shape, k = WORKLOADS[workload]
    deg = np.diff(ptr)
    m, nnz = len(ptr) - 1, int(ptr[-1])
    flushed = bytes_min(m, nnz, k) < 2 * L2_BYTES
    return {
        "workload": workload, "graph": shape, "num_v": m, "nnz": nnz, "K": k,
        "max_row_nnz": int(deg.max()), "mean_row_nnz": round(float(deg.mean()), 2),
        "p50_row_nnz": int(np.percentile(deg, 50)), "p99_row_nnz": int(np.percentile(deg, 99)),
        "empty_rows": int((deg == 0).sum()),
        "l2": "GPU arm: L2 flushed (256 MiB write) between iterations" if flushed
              else "GPU arm: inputs larger than L2 (col/val + B re-streamed every step)",
    }


# ---- evidence files written by the capture scripts (never typed in by hand) ------------------------------------------

KERNEL_SOURCES = ("hpc_b200/csrc/spmm_kernels.cu", "hpc_b200/csrc/preprocess.cu", "hpc_b200/csrc/common.h")


def kernel_source_sha16():
    h = hashlib.sha256()
    for rel in KERNEL_SOURCES:
        h.update(open(os.path.join(ROOT, rel), "rb").read())
    return h.hexdigest()[:16]


def ncu_record(workload):
    """profiles/r02_ncu_<workload>.json (tools/ncu_summarise.py) if it was captured at the current kernel sources."""
    path = os.path.join(ROOT, "profiles", f"r02_ncu_{workload}.json")
    try:
        d = json.load(open(path))
    except Exception:
        return None, "no capture"
    if d.get("kernel_source_sha16") != kernel_source_sha16():
        return None, f"stale (captured at kernel sources {d.get('kernel_source_sha16')})"
    return d, os.path.relpath(path, ROOT)


def l2_gather_peak():
    """Measured L2 -> SM ceiling for whole-row gathers (tools/l2_gather_peak.cu), GB/s by row size."""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "r02_l2_gather_peak.json")))
    except Exception:
        return None


class ClockSampler:
    """SM clock + throttle reasons during the timed region (pynvml, 50 ms period)."""

    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nv = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self._nv = None

    def _loop(self):
        nv = self._nv
        names = {
            "hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
            "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
            "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
            "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4),
        }
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            self._stop.wait(0.05)

    def __enter__(self):
        if self._nv:
            self._thread = threading.Thread(target=self._loop, daemon=True)
            self._thread.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self._thread:
            self._thread.join()

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": 0}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ---- reference arm (host CPU; no product kernel is loaded) ---------------------------------------------------------

def host_gen_named_graph(shape, threads):
    """The graph generator from the host-only library (graph.cpp alone), without importing the hpc_b200 package."""
    spec = importlib.util.spec_from_file_location("_spmm_b200_shapes", os.path.join(ROOT, "hpc_b200", "shapes.py"))
    shapes = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(shapes)
    g = ctypes.CDLL(os.path.join(ROOT, "hpc_b200", "libspmm_b200_graph.so"))
    g.spmm_b200_last_error.restype = ctypes.c_char_p
    g.spmm_b200_gen_graph.argtypes = ([ctypes.c_int, ctypes.c_longlong] + [ctypes.c_int] * 5 +
                                      [ctypes.c_uint64, ctypes.c_void_p, ctypes.c_void_p])
    g.spmm_b200_set_host_threads(int(threads))
    nv, nnz, mx, tk, zp, lp, win = shapes.GRAPH_SHAPES[shape]
    ptr, idx = np.empty(nv + 1, np.int32), np.empty(nnz, np.int32)
    rc = g.spmm_b200_gen_graph(nv, nnz, mx, tk, zp, lp, win, SEED, ptr.ctypes.data, idx.ctypes.data)
    if rc:
        raise RuntimeError(g.spmm_b200_last_error().decode())
    return ptr, idx


def cpu_sample(ptr, idx, k, seconds, nthreads=0):
    """Time the CPU oracle on a bounded prefix of rows; returns (gflops, description, cores, s per pass, nnz)."""
    from oracle import cpu as O
    m, nnz = len(ptr) - 1, int(ptr[-1])
    val = O.fill_normal(nnz, SEED, 1)
    b = O.fill_normal(m * k, SEED, 2)
    out = np.zeros(m * k, np.float32)
    # all the cores this process may use (torchrun exports OMP_NUM_THREADS=1, which would hide them)
    cores = nthreads or max(O.num_threads(), len(os.sched_getaffinity(0)))

    def run(rows):
        t = time.perf_counter()
        O.spmm_f32(ptr, idx, val, b, k, 0, rows, False, cores, out)
        return time.perf_counter() - t

    # calibrate on ~1% of the nonzeros, then size the sample for `seconds`: a row prefix when the
    # whole graph would take longer, otherwise the whole graph repeated
    r1 = int(np.searchsorted(ptr, max(1, nnz // 100), side="left"))
    r1 = max(1, min(m, r1))
    run(r1)
    t1 = run(r1)
    rate = 2.0 * int(ptr[r1]) * k / max(t1, 1e-9)
    want_nnz = min(nnz, int(rate * seconds / (2.0 * k)))
    rows = int(np.searchsorted(ptr, want_nnz, side="left"))
    rows = max(r1, min(m, rows))
    snnz = int(ptr[rows])
    reps, t = 0, 0.0
    while reps == 0 or (rows == m and t < seconds and reps < 10000):
        t += run(rows)
        reps += 1
    desc = f"rows [0,{rows}) of {m} ({snnz} of {nnz} nnz) x {reps} passes, {t:.2f} s"
    return 2.0 * snnz * k * reps / t / 1e9, desc, cores, t / reps, snnz


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    shape, k = WORKLOADS[args.workload]
    ptr, idx = host_gen_named_graph(shape, len(os.sched_getaffinity(0)))
    nnz = len(idx)
    per_step = max(1.0, min(20.0, 150.0 / max(1, args.steps + args.warmup)))
    vals, desc, cores = [], "", 0
    for s in range(args.warmup + args.steps):
        g, desc, cores, t, snnz = cpu_sample(ptr, idx, k, per_step)
        if s >= args.warmup:
            vals.append((g, t, snnz))
    gf = float(np.mean([v[0] for v in vals]))
    ms_full = 2.0 * nnz * k / (gf * 1e9) * 1e3
    line = {
        "impl": "reference", "metric": "spmm_gflops", "value": round(gf, 3), "unit": "GFLOP/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms_full, 3),
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.workload, ptr),
        "note": "ms_per_step extrapolates the sampled rate to the full graph",
        "cpu_baseline": {"value": round(gf, 3), "unit": "GFLOP/s", "cores": cores, "kind": "port",
                         "sample": desc + " per step (OpenMP restatement of spmm_ref.cu:3-17; the reference has no CPU path)"},
        "e2e": {"value": round(gf, 3), "unit": "GFLOP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ---- GPU arm ---------------------------------------------------------------------------------------------------------

class Ctx:
    """torch / torch.distributed / device of this rank."""

    def __init__(self):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device (the engine has no CPU path)")
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        if self.world > 1:
            # one process per GPU: run on the cores next to this GPU, so that the pinned host buffers of the host-buffer
            # call are allocated NUMA-local to its PCIe link (what `numactl` would do around each rank)
            try:
                import pynvml
                pynvml.nvmlInit()
                pynvml.nvmlDeviceSetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(self.local))
            except Exception:
                pass
        if self.world > 1:
            # keep stdout to the one JSON line: whatever NCCL prints while it initialises ("NCCL version ..." is a
            # bare printf at NCCL_DEBUG=VERSION) is sent to stderr by pointing fd 1 at fd 2 for the duration
            sys.stdout.flush()
            saved_fd = os.dup(1)
            os.dup2(2, 1)
            try:
                dist.init_process_group("nccl", device_id=self.dev)
                dist.barrier()
                torch.cuda.synchronize()
            finally:
                sys.stdout.flush()
                os.dup2(saved_fd, 1)
                os.close(saved_fd)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, values):
        t = self.torch.tensor([float(v) for v in values], dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return [float(x) for x in t]

    def gather_over_ranks(self, value):
        t = self.torch.tensor([float(value)], dtype=self.torch.float64, device=self.dev)
        if self.world == 1:
            return [float(value)]
        out = [self.torch.zeros_like(t) for _ in range(self.world)]
        self.dist.all_gather(out, t)
        return [float(x[0]) for x in out]

    def sum_i64(self, value):
        t = self.torch.tensor([int(value)], dtype=self.torch.int64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return int(t[0])


def bits_checksum(t):
    """Order-independent exact checksum: sum of the fp32 bit patterns as integers (mod 2^64). Equal across any
    partition of the rows iff the same multiset of output words was produced."""
    import torch
    return int(t.view(torch.int32).to(torch.int64).sum())


def timed_steps(ctx, fn, steps, flush):
    """K steps, device time per step by CUDA events on the launching stream; -> per-step ms (this rank)."""
    torch = ctx.torch
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for a, b in evs:
        if flush is not None:
            flush.zero_()          # L2 flush between iterations, outside the event pair
        a.record()
        fn()
        b.record()
    ctx.barrier()
    return np.asarray([a.elapsed_time(b) for a, b in evs])


def dump_outputs(ctx, sh, vout, directory):
    """--dump-outputs: C = A·B as a caller of the timed path receives it, written as DIR/C.npy (float32, one row of C
    per line) with the row numbers in DIR/C_rows.npy (float64). A C larger than DUMP_BYTES is a fixed, seeded sample
    of its rows, so that two builds run with the same arguments can be compared output for output. With N > 1 the
    ranks' row blocks are all-gathered first (collective: every rank calls this)."""
    torch = ctx.torch
    m, k = sh.num_v, sh.feat
    full = vout
    if ctx.world > 1:
        full = torch.empty(m * k, dtype=torch.float32, device=ctx.dev)
        sh.allgather(vout, full)
    if ctx.rank != 0:
        return
    n = min(m, DUMP_BYTES // (4 * k + 8))
    rows = np.arange(m) if n == m else np.sort(np.random.default_rng(SEED).choice(m, n, replace=False))
    c = full[: m * k].view(m, k)[torch.from_numpy(rows).to(ctx.dev)].cpu().numpy()
    os.makedirs(directory, exist_ok=True)
    np.save(os.path.join(directory, "C.npy"), c)
    np.save(os.path.join(directory, "C_rows.npy"), rows.astype(np.float64))


def build_sharded(ctx, H, shape, k, opts, graph=None):
    """Graph, nnz-balanced row partition (SURVEY.md §8e), this rank's operator over its block with B replicated."""
    from hpc_b200.dist import ShardedSpMM
    torch = ctx.torch
    H.set_host_threads(max(1, len(os.sched_getaffinity(0)) // ctx.world))   # the generator's share of the host cores
    ptr, idx = graph if graph is not None else H.gen_named_graph(shape, SEED)
    m, nnz = len(ptr) - 1, len(idx)
    val = torch.empty(nnz, dtype=torch.float32, device=ctx.dev)
    H.fill_normal(val, SEED, 1)
    sh = ShardedSpMM(ptr, idx, val, k, device=ctx.dev, **opts)
    del val
    vin = torch.empty(m * k, dtype=torch.float32, device=ctx.dev)
    H.fill_normal(vin, SEED, 2)
    vout = torch.empty(max(1, sh.local_rows * k), dtype=torch.float32, device=ctx.dev)
    torch.cuda.synchronize(ctx.dev)   # the input fills are queued kernels: keep them out of the preprocess clock
    t0 = time.perf_counter()
    sh.preprocess(vin, vout)
    torch.cuda.synchronize(ctx.dev)
    first_s = time.perf_counter() - t0
    # the first plan build of a process also pays CUDA's lazy kernel loading and the first big cudaMalloc / pinned
    # staging allocations; the same call again (the plan is rebuilt from scratch) is what every later operator costs
    t0 = time.perf_counter()
    sh.preprocess(vin, vout)
    torch.cuda.synchronize(ctx.dev)
    prep_s = time.perf_counter() - t0
    return ptr, idx, sh, vin, vout, (prep_s, first_s)


def quick_measure(ctx, H, shape, k, steps=10, warmup=3, checksum=False, graph=None):
    """Kernel-only numbers for one more BASELINE config on the same GPU(s) (L2 flushed between iterations when the
    working set is small)."""
    torch = ctx.torch
    ptr, idx, sh, vin, vout, prep_s = build_sharded(ctx, H, shape, k, {}, graph)
    m, nnz = len(ptr) - 1, len(idx)
    lm = sh.local_rows
    e0, e1 = sh.part.nnz_range(ctx.rank)
    flush = torch.empty(2 * L2_BYTES, dtype=torch.uint8, device=ctx.dev) if bytes_min(lm, e1 - e0, k, m) < 2 * L2_BYTES else None
    for _ in range(warmup):
        if flush is not None:
            flush.zero_()
        sh.run(vin, vout)
    ctx.barrier()
    ts = timed_steps(ctx, lambda: sh.run(vin, vout), steps, flush)
    tw = timed_steps(ctx, lambda: sh.run(vin, vout), steps, None)   # the reference's protocol: back-to-back, L2-warm (util.h:141-151)
    ms, ms_warm = ctx.max_over_ranks([ts.mean(), tw.mean()])
    out = {"workload": f"{shape}_k{k}", "num_v": m, "nnz": nnz, "K": k, "n_gpus": ctx.world, "ms_per_step": round(ms, 5),
           "ms_per_step_l2_warm": round(ms_warm, 5), "gflops": round(2.0 * nnz * k / ms / 1e6, 1),
           "launches_per_step": sh.op.launches_per_run, "preprocess_s": round(prep_s[0], 4),
           "preprocess_first_call_s": round(prep_s[1], 4),
           "l2": "flushed between iterations" if flush is not None else "inputs larger than L2"}
    if ctx.world == 1:
        peak, _ = measured_peaks()
        bm = bytes_min(m, nnz, k)
        out.update({"hbm_gbs_bytes_min": round(bm / ms / 1e6, 1), "roofline_frac": round(bm / ms / 1e6 / peak, 4),
                    "gather_gbs": round(bytes_gather(m, nnz, k) / ms / 1e6, 1)})
    if checksum:
        out["checksum_u64"] = ctx.sum_i64(bits_checksum(vout[: lm * k]) if lm * k else 0) & 0xFFFFFFFFFFFFFFFF
    return out, (ptr, idx, sh, vin, vout)


def stacked_layers(ctx, H, ptr, idx, sh, vin, vout, k, iters=3):
    """BASELINE config 5: two stacked SpMM layers over the ranks, the all-gather of C done (a) by NCCL all-gather-v and
    (b) by the kernel's own epilogue (peer / NVLS multicast stores, no collective). Bit-compared."""
    torch, dist = ctx.torch, ctx.dist
    from hpc_b200.dist import ShardedSpMM
    m = len(ptr) - 1
    full1 = torch.empty(m * k, device=ctx.dev)
    full2 = torch.empty(m * k, device=ctx.dev)

    def two_layers_nccl():
        sh.run(vin, vout)
        sh.allgather(vout, full1)
        sh.run(full1, vout)
        sh.allgather(vout, full2)

    def timed(fn):
        fn()
        ctx.barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(iters):
            fn()
        b.record()
        ctx.barrier()
        return ctx.max_over_ranks([a.elapsed_time(b) / iters])[0]

    t_spmm = timed(lambda: sh.run(vin, vout))
    t_ag = timed(lambda: sh.allgather(vout, full1))
    t_nccl = timed(two_layers_nccl)
    sum1, sum2 = bits_checksum(full1), bits_checksum(full2)

    val = torch.empty(len(idx), dtype=torch.float32, device=ctx.dev)
    H.fill_normal(val, SEED, 1)
    shf = ShardedSpMM(ptr, idx, val, k, device=ctx.dev)
    del val
    bufs = shf.enable_fused_gather(n_buffers=2)
    local_f = torch.empty(max(1, shf.local_rows * k), device=ctx.dev)
    shf.preprocess(vin, local_f)

    def two_layers_fused():
        c1 = shf.run_fused(vin, local_f, buffer=0)
        return shf.run_fused(c1, local_f, buffer=1)

    for b in bufs:
        b.fill_(float("nan"))
    ctx.barrier()
    two_layers_fused()
    ctx.barrier()
    ok = int(torch.equal(bufs[0], full1)) + 2 * int(torch.equal(bufs[1], full2))
    oks = torch.tensor([ok], device=ctx.dev)
    dist.all_reduce(oks, op=dist.ReduceOp.MIN)
    t_fused = timed(two_layers_fused)
    ingress = 4 * (m - shf.local_rows) * k      # bytes every rank must receive per layer
    t_link = ingress / NVLINK_PEER_GBS / 1e6    # ms at the measured peer rate
    out = {
        "layers": 2, "parity": int(oks[0]) == 3, "layer1_bit_equal": bool(int(oks[0]) & 1), "layer2_bit_equal": bool(int(oks[0]) & 2),
        "multicast": bool(shf._use_mc), "ms_spmm_only": round(t_spmm, 4), "ms_allgather_nccl": round(t_ag, 4),
        "ms_nccl": round(t_nccl, 4), "ms_fused": round(t_fused, 4),
        "nvlink_ingress_bytes_per_rank_per_layer": ingress,
        "nvlink_gbs_nccl_allgather": round(ingress / t_ag / 1e6, 1),
        "nvlink_gbs_fused_layer": round(ingress / (t_fused / 2) / 1e6, 1),
        "nvlink_peak_gbs": NVLINK_PEER_GBS, "ms_nvlink_floor_per_layer": round(t_link, 4),
        "binding": "nvlink_ingress" if t_link > t_spmm else "kernel",
        "fused_frac_of_binding": round(max(t_link, t_spmm) / (t_fused / 2), 4),
        "checksum_u64_layer1": sum1 & 0xFFFFFFFFFFFFFFFF, "checksum_u64_layer2": sum2 & 0xFFFFFFFFFFFFFFFF,
    }
    shf.close()
    return out


def run_b200(args):
    ctx = Ctx()
    torch, dist = ctx.torch, ctx.dist
    import hpc_b200 as H
    rank, world, dev = ctx.rank, ctx.world, ctx.dev
    if world != args.gpus and rank == 0:
        print(f"bench.py: --gpus {args.gpus} but WORLD_SIZE={world}; using {world}", file=sys.stderr)

    shape, k = WORKLOADS[args.workload]
    opts = {o.split('=')[0]: int(o.split('=')[1]) for o in args.opt}
    ptr, idx, sh, vin, vout, prep_s = build_sharded(ctx, H, shape, k, opts)
    op = sh.op
    m, nnz = len(ptr) - 1, len(idx)
    lm = sh.local_rows
    e0, e1 = sh.part.nnz_range(rank)
    lnnz = e1 - e0
    info = op.plan_info()

    working_set = bytes_min(lm, lnnz, k, b_rows=m)
    flush = torch.empty(2 * L2_BYTES, dtype=torch.uint8, device=dev) if working_set < 2 * L2_BYTES else None

    for _ in range(args.warmup):
        if flush is not None:
            flush.zero_()
        sh.run(vin, vout)
    ctx.barrier()

    # ---- timed region: K steps, device time by CUDA events on the launching stream ----------
    with ClockSampler(ctx.local) as clocks:
        ctx.barrier()
        wall0 = time.perf_counter()
        step_ms = timed_steps(ctx, lambda: sh.run(vin, vout), args.steps, flush)
        wall = time.perf_counter() - wall0
    if args.dump_outputs:
        dump_outputs(ctx, sh, vout, args.dump_outputs)
    ms_per_step, ms_min = ctx.max_over_ranks([step_ms.mean(), step_ms.min()])
    per_rank_ms = ctx.gather_over_ranks(step_ms.mean())
    launches = op.launches_per_run * args.steps
    dev_sum = bits_checksum(vout[: lm * k]) if lm * k else 0

    # ---- the same step back to back for >= 2 s (the reference's protocol is 31 back-to-back runs, util.h:141-151):
    # sustained clocks and power, L2-warm ----------------------------------------------------------------------------
    n_sus = int(max(20, min(20000, args.sustain_seconds * 1e3 / max(ms_per_step, 1e-3))))
    with ClockSampler(ctx.local) as sus_clocks:
        ctx.barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(n_sus):
            sh.run(vin, vout)
        b.record()
        ctx.barrier()
    sus_ms = ctx.max_over_ranks([a.elapsed_time(b) / n_sus])[0]

    # ---- the kernel's own launch duration (events inside the C ABI, around the launch) --------
    kms = []
    for _ in range(max(3, min(10, args.steps))):
        if flush is not None:
            flush.zero_()
        kms.append(op.run_profiled(vin, vout))
    kernel_ms = float(np.mean(kms))
    n_launch = max(1, op.launches_per_run)   # of the device-resident run (the host-buffer calls below launch per column block)

    # ---- e2e: host buffers through the C ABI, H2D + D2H inside the timed region -------------
    e2e_steps = max(3, min(args.steps, 10))
    h_out = torch.empty(max(1, lm * k), dtype=torch.float32).pin_memory()
    if world == 1:
        h_in = torch.empty(m * k, dtype=torch.float32).pin_memory()
        h_in.copy_(vin.cpu())
        # the host-buffer call gets its own operator over the same CSR, with the column blocks laid out for it (option
        # host_bands: a large last block, whose pass is bound by the PCIe transfer of C anyway)
        host_op = H.SpMMB200(op.g, k, host_bands=1, **opts)
        host_op.preprocess(vin, vout)
        # what the host-buffer call must reproduce bit for bit: the same operator run on device-resident buffers (rows split
        # into segments associate differently under another block layout, so the main operator's bits are not the yardstick)
        ref_out = torch.empty_like(vout)
        host_op.run(vin, ref_out)
        torch.cuda.synchronize()
        host_ref_sum = bits_checksum(ref_out[: lm * k])
        del ref_out
        call = lambda: host_op.run_host(h_in, h_out)  # H2D(B) -> kernels -> C rows stored to the host -> stream sync
        h2d = 4 * m * k
        call_name = ("spmm_b200_run_host (pinned B in, C out; CSR + plan resident, as in the reference harness; plan option "
                     "host_bands = 1)")
    else:
        sh.enable_sharded_host_io()
        h_in = torch.empty(m * k, dtype=torch.float32).pin_memory()   # B on the host; this rank reads only its share of it
        h_in.copy_(vin.cpu())
        call = lambda: sh.run_host_sharded(h_in, h_out)   # H2D(B share) -> NVLink replicate -> kernels -> C block out
        h2d = call()                                      # bytes this rank copies per call, counted by the library
        call_name = ("spmm_b200_run_host_sharded (each rank uploads 1/N of every ~48 MB chunk of B and stores it into every rank's copy "
                     f"over NVLink [{'multimem.st' if sh.rep_multicast else 'peer stores'}], per-chunk flag barrier overlapped with "
                     "the column-block passes, final rows stored straight into the pinned C block)")
    for _ in range(2):
        call()
    ctx.barrier()
    te = time.perf_counter()
    for _ in range(e2e_steps):
        call()
    ctx.barrier()
    e2e_ms = ctx.max_over_ranks([(time.perf_counter() - te) / e2e_steps * 1e3])[0]
    e2e_sum = bits_checksum(h_out[: lm * k]) if lm * k else 0
    same = ctx.sum_i64(int(e2e_sum == (host_ref_sum if world == 1 else dev_sum))) == world
    checksum = ctx.sum_i64(dev_sum) & 0xFFFFFFFFFFFFFFFF
    h2d_all = ctx.sum_i64(h2d)
    if not same:
        raise SystemExit("bench.py: the host-buffer call and the device-resident run disagree (checksum of C)")

    line = None
    if rank == 0:
        flops = 2.0 * nnz * k
        peak, peak_src = measured_peaks()
        total_bytes = bytes_min(lm, lnnz, k, b_rows=m)
        ncu, ncu_src = ncu_record(args.workload) if world == 1 else (None, "captures are single-GPU")
        line = {
            "metric": "spmm_gflops", "value": round(flops / ms_per_step / 1e6, 2), "unit": "GFLOP/s",
            "n_gpus": world, "steps": len(step_ms), "warmup": args.warmup, "ms_per_step": round(ms_per_step, 5),
            "ms_per_step_min": round(ms_min, 5), "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": workload_config(args.workload, ptr),
            "run": {
                "partition": f"rows by nnz over {world} rank(s), B replicated, no collective",
                "plan": {kk: info[kk] for kk in ("seg_len", "kslice", "n_slices", "lanes", "vec", "n_col_blocks", "n_light", "n_heavy", "n_seg",
                                                 "persistent", "n_row_groups", "n_tickets")},
                "preprocess_s": round(prep_s[0], 4), "preprocess_first_call_s": round(prep_s[1], 4),
                "preprocess_note": "preprocess_s = the plan rebuilt by a second preprocess call; first call of the process adds lazy kernel loading and first allocations",
                "per_rank_ms": [round(x, 5) for x in per_rank_ms],
                "kernel_source_sha16": kernel_source_sha16(),
            },
            "sustained": {"ms_per_step": round(sus_ms, 5), "iters": n_sus, "seconds": round(sus_ms * n_sus / 1e3, 2),
                          "gflops": round(flops / sus_ms / 1e6, 2), "clocks": sus_clocks.summary(),
                          "note": "back-to-back runs, inputs unchanged (L2-warm), max over ranks"},
            "hbm_gbs_bytes_min": round(total_bytes / ms_per_step / 1e6, 1),
            "gather_gbs": round(bytes_gather(lm, lnnz, k) / ms_per_step / 1e6, 1),
            "roofline": {
                "bound": "hbm", "kernel": "spmm_kernel", "launches_per_step": n_launch,
                "achieved": round(total_bytes / kernel_ms / 1e6, 1), "peak": peak, "unit": "GB/s",
                "frac": round(total_bytes / kernel_ms / 1e6 / peak, 4),
                "traffic": ncu.get("dram_bytes_per_launch") if ncu else None,
                "l2_hit_pct_ncu": ncu.get("l2_hit_pct") if ncu else None,
                "ncu_source": ncu_src,
                "peak_source": peak_src, "kernel_ms": round(kernel_ms / n_launch, 5),
                "algorithmic_bytes": int(total_bytes // n_launch),
                "gather_gbs": round(bytes_gather(lm, lnnz, k) / kernel_ms / 1e6, 1),
                "binding": binding_bound(k, bytes_gather(lm, lnnz, k) / kernel_ms / 1e6, kernel_ms / n_launch, peak, ncu),
                "note": "per launch (equal shares of the step when there are several); rank 0's partition; algorithmic bytes = "
                        "ptr+col+val+B once+C once (SURVEY.md 8d). The binding bound is the L2->SM gather of B rows (or HBM when B "
                        "is far larger than L2), not compulsory bytes: see DESIGN.md section 3",
            },
            "e2e": {"value": round(flops / e2e_ms / 1e6, 2), "unit": "GFLOP/s", "ms_per_step": round(e2e_ms, 4),
                    "h2d_bytes_per_step": int(h2d_all), "d2h_bytes_per_step": 4 * m * k,
                    "h2d_bytes_per_step_rank0": int(h2d), "d2h_bytes_per_step_rank0": 4 * lm * k, "steps": e2e_steps,
                    "call": call_name, "matches_device_run": bool(same), "checksum_u64": checksum},
            "gpu_launches": int(launches),
            "clocks": clocks.summary(),
            "wall_s_timed_region": round(wall, 4),
        }
    # the buffers of the main workload are no longer needed
    if world == 1:
        host_op.close()
        del host_op
    sh.close()
    del sh, op, vin, vout, h_in, h_out, flush
    torch.cuda.empty_cache()

    if not args.no_also:
        also = []
        if world == 1:
            # the other BASELINE configs, kernel-only, so that one line covers K=32 and K=256 and the products shape
            for wl in ("reddit_k32", "arxiv_k32", "arxiv_k256", "products_k256"):
                if wl != args.workload:
                    sh_, k_ = WORKLOADS[wl]
                    # the metric is quoted at K = 32 and 256: the main graph again at the other width reuses the generated CSR
                    r, keep = quick_measure(ctx, H, sh_, k_, checksum=True, graph=(ptr, idx) if sh_ == shape else None)
                    keep[2].close()
                    del keep
                    torch.cuda.empty_cache()
                    also.append(r)
        elif args.workload != "products_k256":
            # BASELINE config 5 under the same launch: products-shaped graph over the ranks, SpMM alone and two stacked
            # layers with the all-gather of C (NCCL vs the kernel's own epilogue)
            r, keep = quick_measure(ctx, H, "products", 256, steps=5, checksum=True)
            r["stacked"] = stacked_layers(ctx, H, *keep, 256)
            keep[2].close()
            also.append(r)
        if rank == 0:
            line["also"] = also
    if rank == 0:
        if world == 1 and not args.no_cpu_baseline:
            gf, desc, cores, _, _ = cpu_sample(ptr, idx, k, args.cpu_seconds)
            line["cpu_baseline"] = {"value": round(gf, 3), "unit": "GFLOP/s", "cores": cores, "kind": "port", "sample": desc}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def binding_bound(k, gather_gbs, kernel_ms_per_launch, peak_hbm, ncu):
    """What actually binds the kernel, from the capture of the current kernel sources (profiles/r02_ncu_*.json) and the
    measured L2 -> SM gather ceiling (profiles/r02_l2_gather_peak.json): the larger of the two fractions."""
    out = {}
    fab = l2_gather_peak()
    if fab:
        key = "row_1024" if k >= 256 else "row_512" if k >= 128 else "row_128"
        if fab.get(key):
            out["l2_fabric"] = {"achieved": round(gather_gbs, 1), "peak": fab[key], "unit": "GB/s", "frac": round(gather_gbs / fab[key], 4),
                                "source": "tools/l2_gather_peak.cu (profiles/r02_l2_gather_peak.json), best rate of random whole-row gathers from an L2-resident buffer"}
    if ncu and ncu.get("dram_bytes_per_launch"):
        a = ncu["dram_bytes_per_launch"] / kernel_ms_per_launch / 1e6
        out["hbm_traffic"] = {"achieved": round(a, 1), "peak": peak_hbm, "unit": "GB/s", "frac": round(a / peak_hbm, 4),
                              "source": "ncu dram bytes per launch / live kernel time"}
    if out:
        out["bound"] = max((kk for kk in out), key=lambda kk: out[kk]["frac"])
    return out or {"bound": "unknown (no capture at the current kernel sources)"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="reddit_k256", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-also", action="store_true", help="skip the numbers of the other configs")
    ap.add_argument("--cpu-seconds", type=float, default=10.0)
    ap.add_argument("--sustain-seconds", type=float, default=2.0)
    ap.add_argument("--opt", action="append", default=[], help="engine option name=value (tuning runs only)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="GPU arm only: write C of the last timed step to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the GPU arm computes; the reference arm times a sample of rows")
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
