"""SDDMM (spmm_b200_sddmm) timing, one JSON line per workload.

    python tools/sddmm_bench.py [--workloads reddit_k256,...] [--steps 20] [--out DIR]

For each workload: the forward run and sddmm on the SAME handle, alternating, CUDA events around each call, L2 flushed
(256 MiB write outside the event pair) before every call when the working set is below 2x L2 (bench.py's rule).
Reported: median ms of both, GFLOP/s = 2 nnz K / time, gathered bytes (one K-float x_col row per nonzero) / time
against the measured L2-resident gather peak (profiles/r02_l2_gather_peak.json), the ratio to run, a chunked torch
baseline for context, and the device name and power limit read in the same process. Every timed output is checked
bit for bit against the CPU restatement on a seeded sample of rows. With --out, line i is also written to
DIR/r03_sddmm_<workload>.json.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import hpc_b200 as H  # noqa: E402
import sddmm_oracle as SO  # noqa: E402

L2_BYTES = 126 << 20
WORKLOADS = {"reddit_k256": ("reddit", 256), "reddit_k32": ("reddit", 32), "products_k256": ("products", 256),
             "arxiv_k32": ("arxiv", 32), "arxiv_k256": ("arxiv", 256)}


def power_limit_w():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        return float(r.stdout.strip().splitlines()[0])
    except Exception:
        return None


def timed(fn, flush):
    if flush is not None:
        flush.zero_()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1)


def torch_baseline(rows, idx, xr, xc, out, slice_len=1 << 22):
    for s in range(0, idx.numel(), slice_len):
        e = min(idx.numel(), s + slice_len)
        out[s:e] = (xr[rows[s:e]] * xc[idx[s:e]]).sum(1)


def bench(name, steps, peaks):
    shape, K = WORKLOADS[name]
    ptr, idx = H.gen_named_graph(shape)
    M, nnz = len(ptr) - 1, len(idx)
    g = H.CSR(M, nnz, torch.from_numpy(ptr).cuda(), torch.from_numpy(idx).cuda(), H.fill_normal(torch.empty(nnz, device="cuda"), 123, 1))
    xr = H.fill_normal(torch.empty(M * K, device="cuda"), 123, 2)
    xc = H.fill_normal(torch.empty(M * K, device="cuda"), 123, 3)
    c = torch.empty(M * K, device="cuda")
    out = torch.empty(nnz, device="cuda")
    op = H.SpMMB200(g, K)
    op.preprocess(xc, c)
    working_set = 4 * (M + 1) + 8 * nnz + 4 * M * K * 2 + 4 * nnz
    flush = torch.empty(2 * L2_BYTES, dtype=torch.uint8, device="cuda") if working_set < 2 * L2_BYTES else None
    for _ in range(3):   # warm-up (the first sddmm after preprocess sets up the band prefix)
        op.run(xc, c)
        op.sddmm(xr, xc, out)
    torch.cuda.synchronize()
    t_run, t_sd = [], []
    for _ in range(steps):
        t_run.append(timed(lambda: op.run(xc, c), flush))
        t_sd.append(timed(lambda: op.sddmm(xr, xc, out), flush))
    # the output of the last timed call against the oracle on a seeded sample of rows
    rng = np.random.default_rng(2024)
    rows_s = np.sort(rng.choice(M, size=min(M, 512), replace=False))
    deg = np.diff(ptr)[rows_s]
    sub_ptr = np.concatenate([[0], np.cumsum(deg)]).astype(np.int32)
    pos = np.concatenate([np.arange(ptr[r], ptr[r + 1]) for r in rows_s]).astype(np.int64)
    xr_h = xr.view(M, K)[torch.from_numpy(rows_s).cuda()].cpu().numpy()
    want = SO.sddmm_f32(sub_ptr, idx[pos], xr_h, xc.cpu().numpy(), K, ftz=True)
    got = out[torch.from_numpy(pos).cuda()].cpu().numpy()
    check = bool(np.array_equal(got.view(np.int32), want.view(np.int32)))
    # chunked torch baseline (context only)
    rows_t = torch.repeat_interleave(torch.arange(M, device="cuda"), torch.from_numpy(np.diff(ptr)).cuda().long())
    idx_t = g.idx.long()
    ob = torch.empty(nnz, device="cuda")
    torch_baseline(rows_t, idx_t, xr.view(M, K), xc.view(M, K), ob)
    t_torch = [timed(lambda: torch_baseline(rows_t, idx_t, xr.view(M, K), xc.view(M, K), ob), flush) for _ in range(3)]
    ms_run, ms_sd, ms_torch = float(np.median(t_run)), float(np.median(t_sd)), float(np.median(t_torch))
    gathered = 4.0 * nnz * K
    peak_key = "row_1024" if K * 4 >= 1024 else "row_128"
    line = {
        "workload": name, "graph": shape, "num_v": M, "nnz": nnz, "K": K, "steps": steps,
        "n_col_blocks": op.plan_info()["n_col_blocks"],
        "sddmm_ms": round(ms_sd, 4), "run_ms": round(ms_run, 4), "ratio_to_run": round(ms_sd / ms_run, 3),
        "sddmm_ms_min": round(min(t_sd), 4), "run_ms_min": round(min(t_run), 4),
        "gflops": round(2.0 * nnz * K / ms_sd / 1e6, 1),
        "gathered_gb": round(gathered / 1e9, 2), "gather_gbs": round(gathered / ms_sd / 1e6, 1),
        "gather_peak_gbs": peaks[peak_key], "gather_peak_key": peak_key,
        "share_of_gather_peak": round(gathered / ms_sd / 1e6 / peaks[peak_key], 3),
        "floor_ms_at_peak": round(gathered / peaks[peak_key] / 1e6, 3),
        "torch_chunked_ms": round(ms_torch, 3),
        "output_check": {"rows_sampled": int(len(rows_s)), "nonzeros": int(len(pos)), "bit_exact_vs_oracle": check},
        "l2": "flushed (256 MiB write) before every call" if flush is not None else "working set larger than 2x L2",
        "device": torch.cuda.get_device_name(), "power_limit_w": power_limit_w(),
    }
    op.close()
    return line


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--workloads", default=",".join(WORKLOADS))
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("sddmm_bench.py needs a CUDA device")
    peaks = json.load(open(os.path.join(ROOT, "profiles", "r02_l2_gather_peak.json")))
    ok = True
    for name in args.workloads.split(","):
        line = bench(name, args.steps, peaks)
        ok &= line["output_check"]["bit_exact_vs_oracle"]
        print(json.dumps(line), flush=True)
        if args.out:
            os.makedirs(args.out, exist_ok=True)
            with open(os.path.join(args.out, f"r03_sddmm_{name}.json"), "w") as f:
                f.write(json.dumps(line, indent=1) + "\n")
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
