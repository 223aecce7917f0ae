"""Edge softmax and graph attention timing, one JSON line per workload.

    python tools/attention_bench.py [--workloads reddit_k256,...] [--steps 20] [--out DIR]

For each workload:
  - edge_softmax and edge_softmax_backward on real scores (sddmm of seeded q, k), alternating with a device copy of
    the same nnz floats (torch copy_, read + write) as the reference rate, CUDA events around each call, the L2
    flushed (256 MiB write outside the event pair) before every call when the working set is below 2x L2. Bytes:
    forward 8 nnz + 4 (M+1), backward 12 nnz + 4 (M+1), copy 8 nnz.
  - one GraphAttention forward + backward step, phase by phase (the calls the module makes, each between events):
    sddmm, softmax, runs (run_values on the forward and the transposed operator); and the same step through the module
    and autograd, timed as a whole.
  - the timed softmax outputs against the CPU restatement on a seeded sample of rows (bit for bit).
  - the device name and power limit, read in the same process.
With --out, line i is also written to DIR/r04_attention_<workload>.json.
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
import softmax_oracle as SM  # noqa: E402

L2_BYTES = 126 << 20
WORKLOADS = {"reddit_k256": ("reddit", 256), "reddit_k32": ("reddit", 32), "products_k256": ("products", 256),
             "arxiv_k256": ("arxiv", 256)}


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


def sample_check(ptr, s, dp, p, ds, seed=2024):
    """p, ds (device) against the oracle on a seeded sample of rows."""
    M = len(ptr) - 1
    rng = np.random.default_rng(seed)
    rows = np.sort(rng.choice(M, size=min(M, 512), replace=False))
    deg = np.diff(ptr)[rows]
    sub_ptr = np.concatenate([[0], np.cumsum(deg)]).astype(np.int32)
    pos = np.concatenate([np.arange(ptr[r], ptr[r + 1]) for r in rows]).astype(np.int64)
    pos_t = torch.from_numpy(pos).cuda()
    s_h, dp_h = s[pos_t].cpu().numpy(), dp[pos_t].cpu().numpy()
    want_p = SM.edge_softmax_f32(sub_ptr, s_h)
    want_ds = SM.edge_softmax_backward_f32(sub_ptr, want_p, dp_h)
    got_p, got_ds = p[pos_t].cpu().numpy(), ds[pos_t].cpu().numpy()
    same = lambda a, b: bool(np.array_equal(a.view(np.int32), b.view(np.int32)))
    return {"rows_sampled": int(len(rows)), "nonzeros": int(len(pos)),
            "forward_bit_exact_vs_oracle": same(got_p, want_p), "backward_bit_exact_vs_oracle": same(got_ds, want_ds)}


def bench(name, steps):
    shape, K = WORKLOADS[name]
    ptr, idx = H.gen_named_graph(shape)
    M, nnz = len(ptr) - 1, len(idx)
    dev = "cuda"
    g = H.CSR(M, nnz, torch.from_numpy(ptr).cuda(), torch.from_numpy(idx).cuda(), H.fill_normal(torch.empty(nnz, device=dev), 123, 1))
    q, k, v, w = (H.fill_normal(torch.empty(M * K, device=dev), 123, 2 + i).reshape(M, K) for i in range(4))
    att = H.GraphAttention(g, K)
    op, t = att._op(), att.transposed()   # both planned
    s = torch.empty(nnz, device=dev)
    op.sddmm(q, k, s)
    dp = H.fill_normal(torch.empty(nnz, device=dev), 123, 7)
    p, ds = torch.empty(nnz, device=dev), torch.empty(nnz, device=dev)
    src, dst = torch.empty(nnz, device=dev), torch.empty(nnz, device=dev)
    src.copy_(s)
    bytes_fwd, bytes_bwd, bytes_copy = 8 * nnz + 4 * (M + 1), 12 * nnz + 4 * (M + 1), 8 * nnz
    flush = torch.empty(2 * L2_BYTES, dtype=torch.uint8, device=dev) if bytes_bwd < 2 * L2_BYTES else None
    for _ in range(3):
        op.edge_softmax(s, p)
        op.edge_softmax_backward(p, dp, ds)
        dst.copy_(src)
    torch.cuda.synchronize()
    t_f, t_b, t_c = [], [], []
    for _ in range(steps):
        t_c.append(timed(lambda: dst.copy_(src), flush))
        t_f.append(timed(lambda: op.edge_softmax(s, p), flush))
        t_b.append(timed(lambda: op.edge_softmax_backward(p, dp, ds), flush))
    check = sample_check(ptr, s, dp, p, ds)

    # one attention step, phase by phase: the calls GraphAttention makes
    out, dout = torch.empty(M, K, device=dev), w
    dalpha, dq, dk, dv = torch.empty(nnz, device=dev), torch.empty_like(q), torch.empty_like(k), torch.empty_like(v)
    phases = [("sddmm", lambda: op.sddmm(q, k, s)), ("softmax", lambda: op.edge_softmax(s, p)),
              ("runs", lambda: op.run_values(p, v, out)),
              ("sddmm", lambda: op.sddmm(dout, v, dalpha)),
              ("runs", lambda: t.run_values(p, dout, dv)), ("softmax", lambda: op.edge_softmax_backward(p, dalpha, ds)),
              ("runs", lambda: op.run_values(ds, k, dq)),
              ("runs", lambda: t.run_values(ds, q, dk))]
    for _, fn in phases:
        fn()
    torch.cuda.synchronize()
    per_step = []
    for _ in range(max(3, steps // 4)):
        acc = {}
        for ph, fn in phases:
            acc[ph] = acc.get(ph, 0.0) + timed(fn, None)
        per_step.append(acc)
    phase_ms = {ph: med([st[ph] for st in per_step]) for ph in per_step[0]}

    qg, kg, vg = (x.clone().requires_grad_(True) for x in (q, k, v))

    def step():
        qg.grad = kg.grad = vg.grad = None
        (att(qg, kg, vg) * w).sum().backward()

    step()
    torch.cuda.synchronize()
    t_step = [timed(step, None) for _ in range(max(3, steps // 4))]
    ms_f, ms_b, ms_c = med(t_f), med(t_b), med(t_c)
    copy_gbs = bytes_copy / ms_c / 1e6
    line = {
        "workload": name, "graph": shape, "num_v": M, "nnz": nnz, "K": K, "steps": steps,
        "softmax_fwd_ms": ms_f, "softmax_bwd_ms": ms_b, "copy_ms": ms_c,
        "softmax_fwd_ms_min": round(min(t_f), 4), "softmax_bwd_ms_min": round(min(t_b), 4),
        "softmax_fwd_gb": round(bytes_fwd / 1e9, 3), "softmax_bwd_gb": round(bytes_bwd / 1e9, 3),
        "softmax_fwd_gbs": round(bytes_fwd / ms_f / 1e6, 1), "softmax_bwd_gbs": round(bytes_bwd / ms_b / 1e6, 1),
        "copy_gbs": round(copy_gbs, 1),
        "fwd_share_of_copy_rate": round(bytes_fwd / ms_f / 1e6 / copy_gbs, 3),
        "bwd_share_of_copy_rate": round(bytes_bwd / ms_b / 1e6 / copy_gbs, 3),
        "attention_step_phase_ms": phase_ms,
        "attention_step_phase_sum_ms": round(sum(phase_ms.values()), 3),
        "attention_step_autograd_ms": med(t_step),
        "output_check": check,
        "l2": "flushed (256 MiB write) before every softmax / copy call" if flush is not None
              else "working set larger than 2x L2",
        "device": torch.cuda.get_device_name(), "power_limit_w": power_limit_w(),
    }
    att.close()
    return line


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--workloads", default=",".join(WORKLOADS))
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("attention_bench.py needs a CUDA device")
    ok = True
    for name in args.workloads.split(","):
        line = bench(name, args.steps)
        ok &= line["output_check"]["forward_bit_exact_vs_oracle"] and line["output_check"]["backward_bit_exact_vs_oracle"]
        print(json.dumps(line), flush=True)
        if args.out:
            os.makedirs(args.out, exist_ok=True)
            with open(os.path.join(args.out, f"r04_attention_{name}.json"), "w") as f:
                f.write(json.dumps(line, indent=1) + "\n")
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
