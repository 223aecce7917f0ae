"""amax reduce (spmm_b200_reduce) and its gradient (spmm_b200_reduce_backward) timing, one JSON line per workload.

    python tools/reduce_bench.py [--workloads reddit_k256,...] [--steps 20] [--out DIR]

For each workload, on the SAME handle and in one process, alternating call by call: the forward run, reduce("amax") with
arg, reduce("amax") without arg, reduce_backward with db only, and reduce_backward with db and dval (on the transposed
operator). CUDA events around each call after a warm-up; for arxiv the L2 is flushed (a 256 MiB write outside the
event pair) before every call, the other workloads' working sets are larger than the L2. Reported: median and minimum
ms of each, the ratio of each median to run's, the B-row gather floor at the measured L2-resident gather peak
(profiles/r02_l2_gather_peak.json), and the device name and power limit read in the same process. The outputs of the
last timed calls are checked bit for bit against the CPU restatement (tests/reduce_oracle.c): vout and arg on 512
seeded rows, db on 512 seeded rows of B (with every entry of those columns of A) and dval on those entries.
With --out, line i is also written to DIR/r05_reduce_<workload>.json.
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
import reduce_oracle as RO  # noqa: E402

L2_BYTES = 126 << 20
# name -> (graph, K, flush the L2 before every call)
WORKLOADS = {"reddit_k256": ("reddit", 256, False), "reddit_k32": ("reddit", 32, False),
             "products_k256": ("products", 256, False), "arxiv_k256": ("arxiv", 256, True)}


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


def check_forward(ptr, idx, val, vin, vout, arg, M, K, rng):
    rows = np.sort(rng.choice(M, size=min(M, 512), replace=False))
    deg = np.diff(ptr)[rows]
    sub_ptr = np.concatenate([[0], np.cumsum(deg)]).astype(np.int32)
    pos = np.concatenate([np.arange(ptr[r], ptr[r + 1]) for r in rows]).astype(np.int64)
    want_v, want_a = RO.reduce_f32(sub_ptr, idx[pos], val[pos], vin, K, "amax")
    sub_to_pos = np.concatenate([pos, [-1]])
    return bool(np.array_equal(vout[rows].view(np.int32), want_v.view(np.int32))
                and np.array_equal(arg[rows], sub_to_pos[want_a]))


def check_backward(ptr, idx, val, vin, dc, arg, db, dval, M, K, rng):
    """db on 512 seeded rows of B: A restricted to the entries of those columns (rows and positions kept in order),
    arg renumbered to the kept positions (anything else matches nothing)."""
    cols = np.sort(rng.choice(vin.shape[0], size=min(vin.shape[0], 512), replace=False))
    keep = np.isin(idx, cols)
    newpos = np.cumsum(keep) - 1
    rows_of = np.repeat(np.arange(M), np.diff(ptr))
    sub_ptr = np.concatenate([[0], np.cumsum(np.bincount(rows_of[keep], minlength=M))]).astype(np.int32)
    a_ok = arg >= 0
    sub_arg = np.where(a_ok, -2, -1).astype(np.int32)
    hit = np.zeros_like(a_ok)
    hit[a_ok] = keep[arg[a_ok]]
    sub_arg[hit] = newpos[arg[hit]]
    want_db, want_dv = RO.reduce_backward_f32(sub_ptr, idx[keep], val[keep], dc, sub_arg, vin, vin.shape[0], K)
    ok_db = np.array_equal(db[cols].view(np.int32), want_db[cols].view(np.int32))
    ok_dv = np.array_equal(dval[keep].view(np.int32), want_dv.view(np.int32))
    return bool(ok_db), bool(ok_dv), int(keep.sum())


def bench(name, steps, peaks):
    shape, K, flush_l2 = WORKLOADS[name]
    ptr, idx = H.gen_named_graph(shape)
    M, nnz = len(ptr) - 1, len(idx)
    g = H.CSR(M, nnz, torch.from_numpy(ptr).cuda(), torch.from_numpy(idx).cuda(),
              H.fill_normal(torch.empty(nnz, device="cuda"), 123, 1))
    b = H.fill_normal(torch.empty(M * K, device="cuda"), 123, 2)
    dc = H.fill_normal(torch.empty(M * K, device="cuda"), 123, 3)
    c = torch.empty(M * K, device="cuda")
    vout = torch.empty(M * K, device="cuda")
    arg = torch.empty(M * K, dtype=torch.int32, device="cuda")
    db = torch.empty(M * K, device="cuda")
    dval = torch.empty(nnz, device="cuda")
    op = H.SpMMB200(g, K)
    op.preprocess(b, c)
    t = op.transposed()
    flush = torch.empty(2 * L2_BYTES, dtype=torch.uint8, device="cuda") if flush_l2 else None
    calls = {
        "run": lambda: op.run(b, c),
        "reduce_arg": lambda: op.reduce("amax", b, vout, arg),
        "reduce_noarg": lambda: op.reduce("amax", b, vout),
        "backward_db": lambda: t.reduce_backward(dc, arg, db=db),
        "backward_db_dval": lambda: t.reduce_backward(dc, arg, db=db, dval=dval, vin=b),
    }
    for _ in range(3):
        for fn in calls.values():
            fn()
    torch.cuda.synchronize()
    times = {k: [] for k in calls}
    for _ in range(steps):
        for k, fn in calls.items():
            times[k].append(timed(fn, flush))
    op.reduce("amax", b, vout, arg)      # the arg the backward read (the no-arg call left vout equal)
    torch.cuda.synchronize()
    rng = np.random.default_rng(2024)
    val = g.val.cpu().numpy()
    bn, dcn = b.cpu().numpy().reshape(M, K), dc.cpu().numpy().reshape(M, K)
    an = arg.cpu().numpy().reshape(M, K)
    fwd_ok = check_forward(ptr, idx, val, bn, vout.cpu().numpy().reshape(M, K), an, M, K, rng)
    db_ok, dv_ok, n_checked = check_backward(ptr, idx, val, bn, dcn, an, db.cpu().numpy().reshape(M, K),
                                             dval.cpu().numpy(), M, K, rng)
    med = {k: float(np.median(v)) for k, v in times.items()}
    gathered = 4.0 * nnz * K
    peak_key = "row_1024" if K * 4 >= 1024 else "row_128"
    line = {
        "workload": name, "graph": shape, "num_v": M, "nnz": nnz, "K": K, "steps": steps,
        "n_col_blocks": op.plan_info()["n_col_blocks"],
        "ms": {k: round(v, 4) for k, v in med.items()},
        "ms_min": {k: round(min(v), 4) for k, v in times.items()},
        "ratio_to_run": {k: round(v / med["run"], 3) for k, v in med.items() if k != "run"},
        "gathered_gb": round(gathered / 1e9, 2), "gather_peak_gbs": peaks[peak_key], "gather_peak_key": peak_key,
        "floor_ms_at_peak": round(gathered / peaks[peak_key] / 1e6, 3),
        "output_check": {"forward_rows_sampled": 512, "forward_bit_exact": fwd_ok, "db_rows_sampled": 512,
                         "db_bit_exact": db_ok, "dval_entries_checked": n_checked, "dval_bit_exact": dv_ok},
        "l2": "flushed (256 MiB write) before every call" if flush is not None else "working set larger than the L2",
        "device": torch.cuda.get_device_name(), "power_limit_w": power_limit_w(),
    }
    t.close()
    op.close()
    return line


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--workloads", default=",".join(WORKLOADS))
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("reduce_bench.py needs a CUDA device")
    peaks = json.load(open(os.path.join(ROOT, "profiles", "r02_l2_gather_peak.json")))
    ok = True
    for name in args.workloads.split(","):
        line = bench(name, args.steps, peaks)
        chk = line["output_check"]
        ok &= chk["forward_bit_exact"] and chk["db_bit_exact"] and chk["dval_bit_exact"]
        print(json.dumps(line), flush=True)
        if args.out:
            os.makedirs(args.out, exist_ok=True)
            with open(os.path.join(args.out, f"r05_reduce_{name}.json"), "w") as f:
                f.write(json.dumps(line, indent=1) + "\n")
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
