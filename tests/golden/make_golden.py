"""Generates tests/golden/golden.{json,npz}: small SpMM cases with stored outputs.

Provenance of the stored outputs: the CPU oracle (oracle/spmm_oracle.c, literal loop order of
PA4/handout/src/spmm_ref.cu:3-17). The reference's implementation is a CUDA kernel; rebuilt
for sm_100a by oracle/Makefile and run on a B200 it reproduced every stored output bit for bit,
which pins these vectors to the reference. Run from the repo root:  python tests/golden/make_golden.py
"""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import cpu as O  # noqa: E402
from oracle import graph_oracle as G  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))

CASES = [
    # name, (M, nnz, max_deg, tail_k, zero_ppm, local_ppm, window), seed, K
    ("tiny_k32", (64, 640, 48, 2, 100000, 500000, 8), 11, 32),
    ("skew_k32", (512, 8192, 400, 3, 50000, 300000, 32), 12, 32),
    ("skew_k256", (256, 4096, 200, 3, 50000, 300000, 16), 13, 256),
    ("odd_k20", (128, 1024, 100, 2, 0, 0, 1), 14, 20),
    ("scalar_k7", (96, 700, 60, 2, 200000, 1000000, 4), 15, 7),
]

if __name__ == "__main__":
    arrays, meta = {}, {"cases": [], "generator": "oracle/graph_oracle.py + oracle/spmm_oracle.c (literal order)"}
    for name, shape, seed, K in CASES:
        ptr, idx = G.gen_graph(*shape, seed)
        val = O.fill_normal(len(idx), seed, 1)
        b = O.fill_normal((len(ptr) - 1) * K, seed, 2)
        out = O.spmm_literal(ptr, idx, val, b, K)
        arrays[f"{name}_ptr"], arrays[f"{name}_idx"], arrays[f"{name}_out"] = ptr, idx, out
        meta["cases"].append({"name": name, "shape": list(shape), "seed": seed, "K": K,
                              "out_sum_f64": float(out.astype(np.float64).sum())})
    np.savez_compressed(os.path.join(HERE, "golden.npz"), **arrays)
    json.dump(meta, open(os.path.join(HERE, "golden.json"), "w"), indent=1)
    print("wrote", len(CASES), "cases,", os.path.getsize(os.path.join(HERE, "golden.npz")), "bytes")
