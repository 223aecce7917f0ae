"""Generates tests/golden/reference.{json,npz}: the record of spmm_kernel_ref's output (PA4/handout/src/spmm_ref.cu:3-17,
built with --use_fast_math, so an in-order FFMA.FTZ chain per output element) for the inputs on which the GPU parity
tests compare the engine with it (tests/test_gpu_parity.py::reference_output), so that a checkout without the
reference's sources still runs those comparisons.

For every case the output is kept as the SHA-256 of its M*K float32 words in row-major order, plus a seeded sample of
rows (and the heaviest rows) as values. reference.json names, per case, what produced it: the kernel itself where
oracle/_ref/libspmm_ref.so is built (oracle/Makefile, from the reference's sources; needs a GPU), otherwise the CPU
restatement of the kernel with flush-to-zero (oracle/spmm_oracle.c: the same chains in the same order). The tests
check the record against the kernel wherever the kernel is built, and against the restatement everywhere.
Inputs regenerate from seeds exactly as the tests build them.
Run from the repo root (needs the built libraries):  python tests/golden/make_reference_golden.py
"""
import hashlib
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import hpc_b200 as H  # noqa: E402
import refshim  # noqa: E402
from oracle import cpu as O  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
SEED = 123
SAMPLE_ROWS, HEAVIEST_ROWS = 12, 4


def named_inputs(shape, K):
    """gen_named_graph + fill_normal(seed 123): stream 1 for the values, stream 2 for B (tests' dev_inputs)."""
    ptr, idx = H.gen_named_graph(shape)
    return ptr, idx, O.fill_normal(len(idx), SEED, 1), O.fill_normal((len(ptr) - 1) * K, SEED, 2)


def subnormal_inputs(K=32):
    """test_subnormal_inputs_flush_like_the_reference: subnormal operands and products that underflow."""
    ptr, idx = H.gen_named_graph("c0")
    M, nnz = len(ptr) - 1, len(idx)
    rng = np.random.default_rng(11)
    val = rng.normal(0, 0.1, nnz).astype(np.float32)
    b = rng.normal(0, 0.1, (M, K)).astype(np.float32)
    b[rng.random((M, K)) < 0.3] = np.float32(1e-40)
    b[rng.random((M, K)) < 0.2] *= np.float32(1e-37)
    val[rng.random(nnz) < 0.2] = np.float32(3e-39)
    return ptr, idx, val, b


CASES = {
    "c0_k32": lambda: (named_inputs("c0", 32), 32),
    "arxiv_k32": lambda: (named_inputs("arxiv", 32), 32),
    "arxiv_k256": lambda: (named_inputs("arxiv", 256), 256),
    "reddit_k256": lambda: (named_inputs("reddit", 256), 256),
    "products_k256": lambda: (named_inputs("products", 256), 256),
    "c0_k32_subnormal": lambda: (subnormal_inputs(32), 32),
}


def sample_rows(ptr):
    m = len(ptr) - 1
    rng = np.random.default_rng(SEED)
    heaviest = np.argsort(-np.diff(ptr), kind="stable")[:HEAVIEST_ROWS]
    return np.unique(np.concatenate([rng.choice(m, min(m, SAMPLE_ROWS), replace=False), heaviest])).astype(np.int64)


def digest(out):
    return hashlib.sha256(memoryview(np.ascontiguousarray(out, np.float32))).hexdigest()


def kernel_output(ptr, idx, val, b, K):
    """spmm_kernel_ref on the device (refshim.ref_spmm) -> [M, K] float32."""
    import torch
    M = len(ptr) - 1
    dev = [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in (ptr, idx, val, np.ravel(b))]
    out = torch.full((max(1, M * K),), float("nan"), device="cuda")
    refshim.ref_spmm(*dev, out, M, len(idx), K)
    return out[: M * K].cpu().numpy().reshape(M, K)


if __name__ == "__main__":
    meta, arrays = {}, {}
    for name, make in CASES.items():
        (ptr, idx, val, b), K = make()
        if refshim.available():
            out, source = kernel_output(ptr, idx, val, b, K), "spmm_kernel_ref (oracle/_ref/libspmm_ref.so)"
        else:
            out, source = O.spmm_f32(ptr, idx, val, b, K, ftz=True), "CPU restatement (oracle/spmm_oracle.c, ftz)"
        rows = sample_rows(ptr)
        arrays[f"{name}_rows"], arrays[f"{name}_out"] = rows, out[rows]
        meta[name] = {"num_v": len(ptr) - 1, "nnz": len(idx), "K": K, "sha256": digest(out), "source": source}
        print(name, meta[name])
    np.savez_compressed(os.path.join(HERE, "reference.npz"), **arrays)
    json.dump(meta, open(os.path.join(HERE, "reference.json"), "w"), indent=1)
    print("wrote", len(CASES), "cases,", os.path.getsize(os.path.join(HERE, "reference.npz")), "bytes")
