"""run on a snapshot plan against run_values on a live plan (option live_values), and the graph-attention step with and
without staging; one JSON line per workload.

    python tools/live_values_bench.py [--workloads reddit_k256,...] [--steps 20] [--out DIR]

For each workload, in one process:
  - run on an option-0 (snapshot) plan and run_values on a live plan of the same graph and options, alternating call by
    call, CUDA events around each call after a warm-up; median and minimum of `steps` calls each, and the outputs of
    the last timed calls compared bit for bit on the device.
  - one graph-attention forward + backward step (sddmm, softmax, aggregate; dalpha, dv, softmax backward, dq, dk), two
    ways, alternating step by step: "staged", the snapshot operators with every run preceded by a value copy and
    refresh_values (what GraphAttention did before live values), and "live", the calls GraphAttention now makes
    (run_values on live operators, nothing staged). Both steps' outputs (out, dq, dk, dv) are compared bit for bit.
For arxiv the L2 is flushed (a 256 MiB write outside the event pair) before every call and step; the other workloads'
working sets are larger than the L2. The device name and power limit are read in the same process.
With --out, line i is also written to DIR/r06_live_values_<workload>.json.
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

import hpc_b200 as H  # noqa: E402

L2_BYTES = 126 << 20
# name -> (graph, K, flush the L2 before every call)
WORKLOADS = {"reddit_k256": ("reddit", 256, False), "reddit_k32": ("reddit", 32, False),
             "products_k256": ("products", 256, False), "arxiv_k256": ("arxiv", 256, True),
             "arxiv_k32": ("arxiv", 32, True)}


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


def med(xs):
    return round(float(np.median(xs)), 4)


def same_bits(a, b):
    return bool(torch.equal(a.contiguous().view(torch.int32), b.contiguous().view(torch.int32)))


def bench(name, steps):
    shape, K, flush_l2 = WORKLOADS[name]
    ptr, idx = H.gen_named_graph(shape)
    M, nnz = len(ptr) - 1, len(idx)
    dev = "cuda"
    d_ptr, d_idx = torch.from_numpy(ptr).to(dev), torch.from_numpy(idx).to(dev)
    x = H.fill_normal(torch.empty(nnz, device=dev), 123, 1)
    q, k, v, w = (H.fill_normal(torch.empty(M * K, device=dev), 123, 2 + i).reshape(M, K) for i in range(4))
    flush = torch.empty(2 * L2_BYTES, dtype=torch.uint8, device=dev) if flush_l2 else None

    # run (snapshot plan holding x) against run_values(x) (live plan)
    buf = x.clone()
    snap = H.SpMMB200(H.CSR(M, nnz, d_ptr, d_idx, buf), K)
    live = H.SpMMB200(H.CSR(M, nnz, d_ptr, d_idx, x), K, live_values=1)
    c_snap, c_live = torch.empty(M, K, device=dev), torch.empty(M, K, device=dev)
    snap.preprocess(v, c_snap)
    live.preprocess(v, c_live)
    for _ in range(3):
        snap.run(v, c_snap)
        live.run_values(x, v, c_live)
    torch.cuda.synchronize()
    t_run, t_val = [], []
    for _ in range(steps):
        t_run.append(timed(lambda: snap.run(v, c_snap), flush))
        t_val.append(timed(lambda: live.run_values(x, v, c_live), flush))
    run_equal = same_bits(c_snap, c_live)
    launches = (snap.launches_per_run, live.launches_per_run)
    plan = live.plan_info(0)

    # the attention step, staged (snapshot operators) and live (GraphAttention's calls)
    snap_t = snap.transposed(K)
    snap_t.preprocess(q, k)
    att = H.GraphAttention(H.CSR(M, nnz, d_ptr, d_idx, x), K)
    op, t = att._op(), att.transposed()
    s, p = torch.empty(nnz, device=dev), torch.empty(nnz, device=dev)
    dalpha, ds = torch.empty(nnz, device=dev), torch.empty(nnz, device=dev)
    res = {m: [torch.empty(M, K, device=dev) for _ in range(4)] for m in ("staged", "live")}

    def staged_run(o, vals, b, c):
        buf.copy_(vals)
        o.refresh_values()
        o.run(b, c)

    def step(mode):
        out, dq, dk, dv = res[mode]
        op.sddmm(q, k, s)
        op.edge_softmax(s, p)
        op.sddmm(w, v, dalpha)
        if mode == "staged":
            staged_run(snap, p, v, out)
            staged_run(snap_t, p, w, dv)
        else:
            op.run_values(p, v, out)
            t.run_values(p, w, dv)
        op.edge_softmax_backward(p, dalpha, ds)
        if mode == "staged":
            staged_run(snap, ds, k, dq)
            staged_run(snap_t, ds, q, dk)
        else:
            op.run_values(ds, k, dq)
            t.run_values(ds, q, dk)

    for _ in range(2):
        step("staged")
        step("live")
    torch.cuda.synchronize()
    t_st, t_lv = [], []
    for _ in range(steps):
        t_st.append(timed(lambda: step("staged"), flush))
        t_lv.append(timed(lambda: step("live"), flush))
    step_equal = all(same_bits(a, b) for a, b in zip(res["staged"], res["live"]))

    ms_run, ms_val = med(t_run), med(t_val)
    line = {
        "workload": name, "graph": shape, "num_v": M, "nnz": nnz, "K": K, "steps": steps,
        "n_col_blocks": plan["n_col_blocks"], "launches_per_run": launches[1],
        "run_ms": ms_run, "run_values_ms": ms_val,
        "run_ms_min": round(min(t_run), 4), "run_values_ms_min": round(min(t_val), 4),
        "run_values_over_run": round(ms_val / ms_run, 4),
        "weight_bytes_per_call_gb": round(4 * nnz * plan["n_slices"] / 1e9, 3),
        "attention_step_staged_ms": med(t_st), "attention_step_live_ms": med(t_lv),
        "attention_step_staged_ms_min": round(min(t_st), 4), "attention_step_live_ms_min": round(min(t_lv), 4),
        "attention_step_saved_ms": round(med(t_st) - med(t_lv), 4),
        "outputs_bit_equal": {"run_vs_run_values": run_equal, "staged_vs_live_step": step_equal},
        "l2": "flushed (256 MiB write) before every call" if flush is not None else "working set larger than the L2",
        "device": torch.cuda.get_device_name(), "power_limit_w": power_limit_w(),
    }
    att.close()
    snap_t.close()
    snap.close()
    live.close()
    return line


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--workloads", default=",".join(WORKLOADS))
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("live_values_bench.py needs a CUDA device")
    ok = True
    for name in args.workloads.split(","):
        line = bench(name, args.steps)
        ok &= all(line["outputs_bit_equal"].values())
        print(json.dumps(line), flush=True)
        if args.out:
            os.makedirs(args.out, exist_ok=True)
            with open(os.path.join(args.out, f"r06_live_values_{name}.json"), "w") as f:
                f.write(json.dumps(line, indent=1) + "\n")
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
