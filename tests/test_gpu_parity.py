"""GPU parity tests (run on the B200 box: pytest -m gpu). Everything goes through the C ABI.

Bar: bit-exact for integer work (plan, panels, partitions, generated inputs) and for every output
row the engine keeps whole (same in-order FMA chain as PA4/handout/src/spmm_ref.cu:10-14);
rows split into segments are re-associated and must satisfy
    |C - C_ref| <= 1e-5 * sum_i |B[idx_i, j] * val_i|
(the north-star's rel 1e-5, taken relative to the magnitude of the summed terms), and the whole
output must pass the reference's own criterion (valid.cu:8 + test_spmm.cu:43).
"""
import hashlib
import json
import os
from types import SimpleNamespace

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

if not torch.cuda.is_available():
    pytest.skip("no CUDA device", allow_module_level=True)

import hpc_b200 as H  # noqa: E402
from conftest import tiny_csr  # noqa: E402
from oracle import cpu as O  # noqa: E402
from oracle import plan_oracle as P  # noqa: E402
import refshim  # noqa: E402

TOL = 1e-5
DEV = "cuda"


def dev_inputs(ptr, idx, K, seed=123, val=None, b=None, b_rows=None):
    M, nnz = len(ptr) - 1, len(idx)
    b_rows = b_rows or M
    d_ptr = torch.from_numpy(np.ascontiguousarray(ptr, np.int32)).to(DEV)
    d_idx = torch.from_numpy(np.ascontiguousarray(idx, np.int32)).to(DEV)
    if val is None:
        d_val = H.fill_normal(torch.empty(nnz, device=DEV), seed, 1)
    else:
        d_val = torch.from_numpy(np.ascontiguousarray(val, np.float32)).to(DEV)
    if b is None:
        vin = H.fill_normal(torch.empty(b_rows * K, device=DEV), seed, 2)
    else:
        vin = torch.from_numpy(np.ascontiguousarray(b, np.float32).ravel()).to(DEV)
    vout = torch.full((max(1, M * K),), float("nan"), device=DEV)
    return H.CSR(M, nnz, d_ptr, d_idx, d_val), vin, vout


def run_engine(ptr, idx, K, val=None, b=None, **opts):
    g, vin, vout = dev_inputs(ptr, idx, K, val=val, b=b)
    op = H.SpMMB200(g, K, **opts)
    op.preprocess(vin, vout)
    op.run(vin, vout)
    torch.cuda.synchronize()
    M = g.num_v
    return op, g, vin, vout, vout[: M * K].cpu().numpy().reshape(M, K)


def check_against_oracle(ptr, idx, K, op, g, vin, got):
    M = g.num_v
    val, b = g.val.cpu().numpy(), vin.cpu().numpy()
    ref = O.spmm_f32(ptr, idx, val, b, K)
    assert not np.isnan(got).any()
    heavy = op.heavy_row_set()
    light = np.asarray([r for r in range(M) if r not in heavy], np.int64)
    assert np.array_equal(got[light].view(np.int32), ref[light].view(np.int32)), "whole rows must be bit-exact"
    ab = O.spmm_abssum(ptr, idx, val, b, K)
    assert np.all(np.abs(got.astype(np.float64) - ref) <= TOL * ab + 1e-30)
    # regression guard, well inside the stated tolerance: re-associated fp32 sums stay within a few ulp of the terms
    assert np.all(np.abs(got.astype(np.float64) - ref) <= 2e-6 * ab + 1e-30)
    # the reference's pass criterion, candidate first (test_spmm.cu:43)
    assert O.validate_float(got, ref) < M * K // 10000 + 1
    return ref


# ---- the oracle is pinned to the reference's own kernel -------------------------------------------

def reference_output(golden_dir, name, ptr, idx, K, g, vin):
    """spmm_kernel_ref's output on the test's device inputs -> [M, K] float32, checked against the stored record of the
    case (tests/golden/make_reference_golden.py: SHA-256 of all M*K words, sample rows). Where oracle/_ref is built the
    kernel itself runs, so the record is checked against the kernel; in a checkout without it the CPU restatement of
    the kernel with flush-to-zero stands in and must reproduce the record bit for bit."""
    M = g.num_v
    if refshim.available():
        out = torch.full((max(1, M * K),), float("nan"), device=DEV)
        refshim.ref_spmm(g.ptr, g.idx, g.val, vin, out, M, g.num_e, K)
        ref = out[: M * K].cpu().numpy().reshape(M, K)
    else:
        ref = O.spmm_f32(ptr, idx, g.val.cpu().numpy(), vin[: M * K].cpu().numpy(), K, ftz=True)
    meta = json.load(open(os.path.join(golden_dir, "reference.json")))[name]
    data = np.load(os.path.join(golden_dir, "reference.npz"))
    assert (M, g.num_e, K) == (meta["num_v"], meta["nnz"], meta["K"]), name
    assert np.array_equal(ref[data[f"{name}_rows"]].view(np.int32), data[f"{name}_out"].view(np.int32)), name
    assert hashlib.sha256(memoryview(np.ascontiguousarray(ref))).hexdigest() == meta["sha256"], name
    return ref


def test_reference_kernel_pins_oracle_and_golden(golden_dir):
    """CPU oracle == stored golden outputs, bitwise, from the device-generated inputs; and where oracle/_ref is built,
    spmm_kernel_ref (unmodified, sm_100a, -O3 --use_fast_math) == both."""
    meta = json.load(open(os.path.join(golden_dir, "golden.json")))
    data = np.load(os.path.join(golden_dir, "golden.npz"))
    for case in meta["cases"]:
        n, K = case["name"], case["K"]
        ptr, idx = data[f"{n}_ptr"], data[f"{n}_idx"]
        g, vin, vout = dev_inputs(ptr, idx, K, seed=case["seed"])
        want = data[f"{n}_out"].view(np.int32).reshape(g.num_v, K)
        ora = O.spmm_f32(ptr, idx, g.val.cpu().numpy(), vin.cpu().numpy(), K, ftz=True)
        assert np.array_equal(ora.view(np.int32), want), n
        if refshim.available():
            refshim.ref_spmm(g.ptr, g.idx, g.val, vin, vout, g.num_v, g.num_e, K)
            got = vout[: g.num_v * K].cpu().numpy().reshape(g.num_v, K)
            assert np.array_equal(got.view(np.int32), want), n


@pytest.mark.parametrize("shape,K", [("c0", 32), ("arxiv", 32), ("arxiv", 256)])
def test_engine_vs_reference_kernel(shape, K, golden_dir):
    """BASELINE configs 0-2: engine vs the reference kernel's output on identical device inputs."""
    ptr, idx = H.gen_named_graph(shape)
    op, g, vin, vout, got = run_engine(ptr, idx, K)
    M = g.num_v
    ref = reference_output(golden_dir, f"{shape}_k{K}", ptr, idx, K, g, vin)
    ref_out = torch.from_numpy(ref.ravel()).to(DEV)
    heavy = op.heavy_row_set()
    light = np.asarray([r for r in range(M) if r not in heavy], np.int64)
    assert np.array_equal(got[light].view(np.int32), ref[light].view(np.int32))
    # the reference's criterion (valid.cu:8), the reference's argument order (test_spmm.cu:43); its own validator where built
    assert O.validate_float(got, ref) < M * K // 10000 + 1
    if refshim.available():
        assert refshim.ref_valid(vout, ref_out, M * K) < M * K // 10000 + 1
    assert H.valid(vout, ref_out, M * K) == O.validate_float(got, ref)
    # and the oracle agrees with the reference's output bit for bit at this size too
    ora = check_against_oracle(ptr, idx, K, op, g, vin, got)
    assert np.array_equal(ora.view(np.int32), ref.view(np.int32))
    op.close()


def test_subnormal_inputs_flush_like_the_reference(golden_dir):
    """The handout is built with --use_fast_math, so spmm_kernel_ref is an FFMA.FTZ chain: subnormal operands and
    results are flushed to zero. The engine is built with -ftz=true and must agree bit for bit on such inputs."""
    ptr, idx = H.gen_named_graph("c0")
    K = 32
    M, nnz = len(ptr) - 1, len(idx)
    rng = np.random.default_rng(11)
    val = rng.normal(0, 0.1, nnz).astype(np.float32)
    b = rng.normal(0, 0.1, (M, K)).astype(np.float32)
    b[rng.random((M, K)) < 0.3] = np.float32(1e-40)                 # subnormal operands
    b[rng.random((M, K)) < 0.2] *= np.float32(1e-37)                # products that underflow
    val[rng.random(nnz) < 0.2] = np.float32(3e-39)
    op, g, vin, vout, got = run_engine(ptr, idx, K, val=val, b=b, seg_len=1 << 20)     # every row whole
    ref = reference_output(golden_dir, "c0_k32_subnormal", ptr, idx, K, g, vin)
    assert np.array_equal(got.view(np.int32), ref.view(np.int32))
    assert np.array_equal(O.spmm_f32(ptr, idx, val, b, K, ftz=True).view(np.int32), ref.view(np.int32))
    assert not np.array_equal(O.spmm_f32(ptr, idx, val, b, K, ftz=False).view(np.int32), ref.view(np.int32))   # the inputs do exercise FTZ
    op.close()


# ---- engine vs oracle -----------------------------------------------------------------------------

def _spmm_instance_cases():
    """One case per reachable spmm_kernel<LANES, VEC, TUNE, FULL> (spmm_kernels.cu launch_lanes), chosen through kslice:
    FULL (K a multiple of a whole lanes x vec x 4 slice) at K = 2 * kslice, and not FULL at a kslice that is not
    lanes x vec x 4 and a K that leaves a partial last slice (LANES = 1 has no such kslice); each with tune 0 and 1 and
    segments short enough to give heavy rows. -> (params, {(K, kslice): (lanes, vec, full)})"""
    cases = [(2 * kslice, kslice, lanes, vec, True) for kslice, lanes, vec in
             ((4, 1, 1), (8, 2, 1), (16, 4, 1), (32, 8, 1), (64, 16, 1), (128, 32, 1), (256, 32, 2))]
    cases += [(K, kslice, lanes, vec, False) for kslice, K, lanes, vec in
              ((8, 20, 2, 1), (12, 28, 4, 1), (24, 52, 8, 1), (48, 100, 16, 1), (96, 196, 32, 1), (192, 388, 32, 2))]
    params, shapes = [], {}
    for K, kslice, lanes, vec, full in cases:
        for tune in (0, 1):
            opts = {"kslice": kslice, "tune": tune, "seg_len": 32}
            params.append(pytest.param("c0", K, opts, id=f"c0-K{K}-kslice{kslice}-tune{tune}"))
            shapes[(K, tuple(sorted(opts.items())))] = (lanes, vec, full)
    return params, shapes


SPMM_INSTANCES, SPMM_INSTANCE_SHAPE = _spmm_instance_cases()


@pytest.mark.parametrize("shape,K,opts", [
    ("c0", 32, {}), ("c0", 32, {"seg_len": 16}), ("c0", 32, {"reorder": 0}), ("c0", 256, {"seg_len": 64, "kslice": 64}),
    ("c0", 256, {"kslice": 128}), ("c0", 64, {}), ("c0", 128, {"block": 128}), ("c0", 512, {}), ("c0", 260, {}),
    ("c0", 100, {}), ("c0", 20, {}), ("c0", 8, {}), ("c0", 4, {}), ("c0", 30, {}), ("c0", 7, {}), ("c0", 1, {}),
    ("arxiv", 32, {}), ("arxiv", 256, {}), ("arxiv", 256, {"kslice": 32, "seg_len": 128}),
    ("c0", 32, {"light_steps": 32}), ("c0", 64, {"light_steps": 1000}), ("arxiv", 32, {"light_steps": 33, "reorder": 0}),
    ("c0", 8, {"light_steps": 40}), ("c0", 4, {"col_blocks": 2}),
    ("c0", 32, {"col_blocks": 3}), ("c0", 256, {"col_blocks": 4, "seg_len": 16}), ("arxiv", 256, {"col_blocks": 5}),
    ("arxiv", 32, {"col_blocks": 2, "reorder": 0}), ("c0", 64, {"col_blocks": 64}),
    ("arxiv", 32, {"tune": 1}), ("arxiv", 256, {"tune": 1}), ("c0", 64, {"tune": 1, "seg_len": 32}), ("c0", 100, {"tune": 1}),
    ("arxiv", 256, {"reorder": 0}), ("arxiv", 32, {"reorder": 1}),
] + SPMM_INSTANCES)
def test_engine_matches_oracle(shape, K, opts):
    ptr, idx = H.gen_named_graph(shape)
    op, g, vin, vout, got = run_engine(ptr, idx, K, **opts)
    want = SPMM_INSTANCE_SHAPE.get((K, tuple(sorted(opts.items()))))
    if want is not None:   # the kernel instantiation the case is there for is the one that ran
        info = op.plan_info()
        lanes, vec, kslice = info["lanes"], info["vec"], info["kslice"]
        assert (lanes, vec, K % (lanes * vec * 4) == 0 and kslice == lanes * vec * 4) == want
        assert info["n_heavy"] > 0
    check_against_oracle(ptr, idx, K, op, g, vin, got)
    op.close()


@pytest.mark.parametrize("shape,K", [("collab", 32), ("ddi", 32), ("youtube", 32), ("am", 32), ("yelp", 32), ("wikikg2", 32),
                                     ("collab", 256), ("ddi", 256), ("am", 256)])
def test_dataset_shapes_strict_parity(shape, K):
    """More of run_all.sh's dataset shapes under the strict bar (bit-exact whole rows, 1e-5 split rows), not only the
    reference's 1e-2 criterion that tests/cpp/run_all.py applies to all 13."""
    ptr, idx = H.gen_named_graph(shape)
    op, g, vin, vout, got = run_engine(ptr, idx, K)
    check_against_oracle(ptr, idx, K, op, g, vin, got)
    op.close()


def test_golden_vectors_through_engine(golden_dir):
    meta = json.load(open(os.path.join(golden_dir, "golden.json")))
    data = np.load(os.path.join(golden_dir, "golden.npz"))
    for case in meta["cases"]:
        n, K = case["name"], case["K"]
        ptr, idx = data[f"{n}_ptr"], data[f"{n}_idx"]
        g, vin, vout = dev_inputs(ptr, idx, K, seed=case["seed"])
        op = H.SpMMB200(g, K, seg_len=1 << 20)      # every row whole => bit-exact with the stored output
        op.preprocess(vin, vout)
        op.run(vin, vout)
        got = vout[: g.num_v * K].cpu().numpy().reshape(g.num_v, K)
        assert np.array_equal(got.view(np.int32), data[f"{n}_out"].view(np.int32).reshape(got.shape)), n
        op.close()


EDGE = {
    "all_rows_empty": ([[], [], [], []], 4),
    "one_by_one": ([[(0, 2.0)]], 1),
    "empty_first_last": ([[], [(0, 1.0), (2, -1.0)], []], 3),
    "duplicate_columns": ([[(1, 1e8), (1, 1.0), (1, -1e8)], [(0, 1.0), (0, 1.0)]], 2),
    "unsorted_columns": ([[(2, 1.0), (0, 2.0), (1, 3.0)], [], [(1, 1.0)]], 3),
}


@pytest.mark.parametrize("name", sorted(EDGE))
@pytest.mark.parametrize("K", [4, 32, 33])
def test_edge_cases(name, K):
    rows, m = EDGE[name]
    ptr, idx, val = tiny_csr(rows)
    rng = np.random.default_rng(5)
    b = rng.normal(0, 1, (m, K)).astype(np.float32)
    op, g, vin, vout, got = run_engine(ptr, idx, K, val=val, b=b)
    ref = O.spmm_literal(ptr, idx, val, b, K)
    assert np.array_equal(got.view(np.int32), ref.view(np.int32))
    op.close()


@pytest.mark.parametrize("length", [255, 256, 257, 511, 513, 10000])
@pytest.mark.parametrize("K", [32, 256])
def test_single_long_row(length, K):
    """Row lengths around the segment size (the student's kBatchSize = 256, spmm_opt.cu:6)."""
    m = 12000
    rng = np.random.default_rng(length)
    cols = np.sort(rng.choice(m, length, replace=False)).astype(np.int32)
    ptr = np.zeros(m + 1, np.int32)
    ptr[4:] = length          # row 3 holds everything
    ptr[m] = length + 1       # plus one entry in the last row
    idx = np.concatenate([cols, [7]]).astype(np.int32)
    op, g, vin, vout, got = run_engine(ptr, idx, K, seg_len=256)
    info = op.plan_info()
    assert info["n_heavy"] == (1 if length > 256 else 0)
    check_against_oracle(ptr, idx, K, op, g, vin, got)
    op.close()


@pytest.mark.parametrize("K", [32, 256, 100])
def test_every_row_heavy(K):
    """No light rows at all (the ddi shape at K=32 is like this): the stream part of the launch is empty."""
    m, d = 37, 300
    rng = np.random.default_rng(7)
    ptr = (np.arange(m + 1) * d).astype(np.int32)
    idx = np.concatenate([np.sort(rng.choice(4096, d, replace=False)) for _ in range(m)]).astype(np.int32)
    ptr_full = np.concatenate([ptr, np.full(4096 - m, ptr[-1], np.int32)])       # square: 4096 rows, the rest empty
    for rows_ptr in (ptr_full,):
        op, g, vin, vout, got = run_engine(rows_ptr, idx, K, seg_len=16)
        assert op.plan_info()["n_heavy"] == m
        check_against_oracle(rows_ptr, idx, K, op, g, vin, got)
        op.close()
    # and with literally zero light rows (rectangular block: 37 rows of a 4096-column matrix)
    g, vin, vout = dev_inputs(ptr, idx, K, b_rows=4096)
    op = H.SpMMB200(g, K, b_rows=4096, seg_len=16)
    op.preprocess(vin, vout)
    info = op.plan_info()
    assert info["n_light"] == 0 and info["n_ltask"] == 0 and info["n_heavy"] == m
    op.run(vin, vout)
    torch.cuda.synchronize()
    got = vout[: m * K].cpu().numpy().reshape(m, K)
    val, b = g.val.cpu().numpy(), vin.cpu().numpy().reshape(4096, K)
    want = np.stack([(b[idx[ptr[r]:ptr[r + 1]]].astype(np.float64) * val[ptr[r]:ptr[r + 1], None]).sum(0) for r in range(m)])
    scale = np.stack([np.abs(b[idx[ptr[r]:ptr[r + 1]]].astype(np.float64) * val[ptr[r]:ptr[r + 1], None]).sum(0) for r in range(m)])
    assert np.all(np.abs(got - want) <= TOL * scale)
    op.close()


def test_nnz_zero_and_empty_graph():
    ptr = np.zeros(6, np.int32)
    idx = np.zeros(0, np.int32)
    op, g, vin, vout, got = run_engine(ptr, idx, 32)
    assert not got.any() and not np.isnan(got).any()
    op.close()
    g = H.CSR(0, 0, torch.zeros(1, dtype=torch.int32, device=DEV), torch.zeros(0, dtype=torch.int32, device=DEV),
              torch.zeros(0, device=DEV))
    op = H.SpMMB200(g, 32)
    z = torch.zeros(1, device=DEV)
    op.preprocess(z, z)
    op.run(z, z)
    torch.cuda.synchronize()
    op.close()


def test_call_protocol_and_idempotence():
    ptr, idx = H.gen_named_graph("c0")
    K = 32
    g, vin, vout = dev_inputs(ptr, idx, K)
    op = H.SpMMB200(g, K, seg_len=64)
    with pytest.raises(H.SpmmB200Error) as e:
        op.run(vin, vout)                 # run before preprocess
    assert e.value.code == -2
    op.preprocess(vin, vout)
    op.run(vin, vout)
    first = vout.clone()
    vout.fill_(float("inf"))              # run must not depend on vout's contents (unlike spmm_opt.cu:34,67-68)
    for _ in range(3):
        op.run(vin, vout)
    assert torch.equal(first, vout)
    # other buffers than the ones given to preprocess, on a non-default stream
    vin2 = H.fill_normal(torch.empty_like(vin), 9, 9)
    vout2 = torch.empty_like(vout)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        op.run(vin2, vout2)
    s.synchronize()
    ref = O.spmm_f32(ptr, idx, g.val.cpu().numpy(), vin2.cpu().numpy(), K)
    ab = O.spmm_abssum(ptr, idx, g.val.cpu().numpy(), vin2.cpu().numpy(), K)
    assert np.all(np.abs(vout2.cpu().numpy().reshape(-1, K).astype(np.float64) - ref) <= TOL * ab + 1e-30)
    # set_feat invalidates the plan
    op.set_feat(16)
    with pytest.raises(H.SpmmB200Error) as e:
        op.run(vin, vout)
    assert e.value.code == -2
    # misaligned vin is refused, not silently mis-read
    op.set_feat(K)
    op.preprocess(vin, vout)
    big = torch.zeros(vin.numel() + 8, device=DEV)
    with pytest.raises(H.SpmmB200Error) as e:
        op.run(big[1:], vout)
    assert e.value.code == -1
    op.close()


def test_plan_memory_is_recycled_and_trimmed():
    """Plan arrays come from the library's retaining memory pool (pool.cu): re-planning on one handle,
    on another stream, destroying and creating operators and trimming the pool in between never changes a bit."""
    ptr, idx = H.gen_named_graph("c0")
    K = 64
    g, vin, vout = dev_inputs(ptr, idx, K)
    op = H.SpMMB200(g, K, col_blocks=3, seg_len=32)
    op.preprocess(vin, vout)
    op.run(vin, vout)
    first = vout.clone()
    s = torch.cuda.Stream()
    for rep in range(3):
        vout.fill_(float("nan"))
        if rep == 1:
            s.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s):          # blocks freed in the legacy stream's order are taken over on another stream
                op.preprocess(vin, vout)
                op.run(vin, vout)
            s.synchronize()
        else:
            op.preprocess(vin, vout)
            op.run(vin, vout)
        assert torch.equal(first, vout)
    op.close()
    H.trim_memory()
    H.trim_memory()                             # nothing left to return: still fine
    op = H.SpMMB200(g, K, col_blocks=3, seg_len=32)
    op.preprocess(vin, vout)
    other = H.SpMMB200(g, K)                    # two live plans next to each other
    vout2 = torch.empty_like(vout)
    other.preprocess(vin, vout2)
    H.trim_memory()                             # live plans stay intact
    vout.fill_(float("nan"))
    op.run(vin, vout)
    other.run(vin, vout2)
    assert torch.equal(first, vout)
    check_against_oracle(ptr, idx, K, other, g, vin, vout2.cpu().numpy().reshape(-1, K))
    op.close()
    other.close()


def test_plain_cuda_malloc_path_without_the_pool():
    """SPMM_B200_POOL=0: the same results with cudaMalloc / cudaFree (the pool is an allocator, nothing else)."""
    import subprocess
    import sys
    code = (
        "import sys, torch, numpy as np; sys.path.insert(0, '.'); import hpc_b200 as H\n"
        "ptr, idx = H.gen_named_graph('c0'); M, nnz, K = len(ptr) - 1, len(idx), 64\n"
        "g = H.CSR(M, nnz, torch.from_numpy(ptr).cuda(), torch.from_numpy(idx).cuda(), H.fill_normal(torch.empty(nnz, device='cuda'), 123, 1))\n"
        "vin = H.fill_normal(torch.empty(M * K, device='cuda'), 123, 2); vout = torch.empty(M * K, device='cuda')\n"
        "op = H.SpMMB200(g, K, col_blocks=3, seg_len=32)\n"
        "for _ in range(2): op.preprocess(vin, vout); op.run(vin, vout)\n"
        "H.trim_memory(); torch.cuda.synchronize()\n"
        "print(int(vout.view(torch.int32).to(torch.int64).sum())); op.close()\n")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sums = []
    for pool in ("0", "1"):
        r = subprocess.run([sys.executable, "-c", code], cwd=root, env={**os.environ, "SPMM_B200_POOL": pool}, capture_output=True, text=True,
                           timeout=300)
        assert r.returncode == 0, r.stderr[-2000:]
        sums.append(int(r.stdout.strip().splitlines()[-1]))
    assert sums[0] == sums[1]


def test_preprocess_rejects_inconsistent_csr():
    """Bad inputs come back as status codes with a message (the reference asserts / exits: data.cu:40-45, util.h:63-84)."""
    ptr, idx = H.gen_named_graph("c0")
    K = 32
    g, vin, vout = dev_inputs(ptr, idx, K)
    bad_ptr = g.ptr.clone()
    bad_ptr[-1] -= 1                                   # ptr[num_v] != num_e
    op = H.SpMMB200(H.CSR(g.num_v, g.num_e, bad_ptr, g.idx, g.val), K)
    with pytest.raises(H.SpmmB200Error) as e:
        op.preprocess(vin, vout)
    assert e.value.code == -1 and "ptr" in str(e.value)
    op.close()
    bad_idx = g.idx.clone()
    bad_idx[12345] = g.num_v                           # column outside B
    op = H.SpMMB200(H.CSR(g.num_v, g.num_e, g.ptr, bad_idx, g.val), K)
    with pytest.raises(H.SpmmB200Error) as e:
        op.preprocess(vin, vout)
    assert e.value.code == -1 and "column" in str(e.value)
    with pytest.raises(H.SpmmB200Error):
        op.run(vin, vout)                              # no plan was built
    op.close()
    dec = g.ptr.clone()
    dec[10], dec[11] = int(dec[11]), int(dec[10])      # a decreasing ptr
    if int(dec[10]) != int(dec[11]):
        op = H.SpMMB200(H.CSR(g.num_v, g.num_e, dec, g.idx, g.val), K)
        with pytest.raises(H.SpmmB200Error):
            op.preprocess(vin, vout)
        op.close()


@pytest.mark.parametrize("opts", [{}, {"col_blocks": 3}])
def test_run_host_matches_device_run(opts):
    """Host-buffer call (with column blocks B is uploaded band by band while earlier passes compute)."""
    ptr, idx = H.gen_named_graph("c0")
    K = 64
    op, g, vin, vout, got = run_engine(ptr, idx, K, **opts)
    h_in = vin.cpu().pin_memory()
    h_out = torch.empty(g.num_v * K).pin_memory()
    for _ in range(3):      # repeated calls reuse the staging buffers and events
        h_out.fill_(float("nan"))
        op.run_host(h_in, h_out)
        assert np.array_equal(h_out.numpy().view(np.int32), got.ravel().view(np.int32))
    info = op.plan_info()
    want = info["n_col_blocks"] * (2 if info["n_col_blocks"] > 1 else 1)   # row halves on two streams
    assert op.run_profiled(vin, vout) > 0 and op.launches_per_run == want
    op.close()


# ---- integer paths: bit-exact -----------------------------------------------------------------------

@pytest.mark.parametrize("shape,seg_len,reorder", [("c0", 0, 1), ("c0", 16, 1), ("c0", 16, 0), ("arxiv", 0, 1), ("arxiv", 100, 1), ("arxiv", 0, 0)])
def test_plan_matches_oracle(shape, seg_len, reorder):
    ptr, idx = H.gen_named_graph(shape)
    g, vin, vout = dev_inputs(ptr, idx, 32)
    op = H.SpMMB200(g, 32, seg_len=seg_len, reorder=reorder)
    op.preprocess(vin, vout)
    info = op.plan_info()
    want = P.plan(ptr, idx, g.val.cpu().numpy(), info["seg_len"], bool(reorder), k4=8, pad=4 * (32 // info["lanes"]))
    got = op.plan_arrays()
    assert info["seg_len"] == (seg_len or P.auto_seg_len(len(idx), 32))
    assert info["kslice"] == P.auto_kslice(g.num_v, 32)
    # natural order: the rows are planned in 16 row groups (tasks cut at the bounds); bucketed order: one group
    assert info["n_row_groups"] == (1 if reorder else 16)
    group_row = None if reorder else P.partition_rows(ptr, info["n_row_groups"])
    want.update(P.light_stream(want, idx, g.val.cpu().numpy(), 32 // info["lanes"], info["light_steps"], k4=8, group_row=group_row))
    want["utask"] = P.unified_tasks(want, want, bool(reorder))
    assert np.array_equal(got["utask"], want["utask"]) and info["n_utask"] == info["n_ltask"] + info["n_seg"]
    total = int(want["light_desc"][:, 2].astype(np.int64).sum()) + len(want["light_desc"])
    assert info["light_steps"] == P.auto_light_steps(32 // info["lanes"], total, info["resident_warps"], len(want["seg_desc"]))
    assert info["resident_warps"] >= 148 * 8
    for k in ("row_perm", "light_desc", "ltask", "lpanel", "heavy_rows", "heavy_seg0", "seg_desc", "seg_hrow", "panel"):
        assert np.array_equal(got[k], want[k]), k
    host = H.plan_host(ptr, 32, seg_len, bool(reorder))
    for k in ("row_perm", "heavy_rows", "heavy_seg0", "seg_desc"):
        assert np.array_equal(host[k], want[k]), k
    op.close()


@pytest.mark.parametrize("shape,K,nb,seg_len", [("c0", 32, 3, 16), ("arxiv", 256, 4, 0), ("c0", 64, 7, 32)])
def test_column_block_plan_matches_oracle(shape, K, nb, seg_len):
    ptr, idx = H.gen_named_graph(shape)
    g, vin, vout = dev_inputs(ptr, idx, K)
    op = H.SpMMB200(g, K, col_blocks=nb, seg_len=seg_len)
    op.preprocess(vin, vout)
    info = op.plan_info(0)
    assert info["n_col_blocks"] == nb
    M = g.num_v
    split = P.split_rows(ptr, idx, nb, M)
    val = g.val.cpu().numpy()
    cpb = -(-M // nb)
    covered = np.zeros(len(idx), np.int32)
    for b in range(nb):
        got = op.plan_arrays(b)
        inf = op.plan_info(b)
        assert (inf["col_begin"], inf["col_end"]) == (b * cpb, min(M, (b + 1) * cpb))
        assert np.array_equal(got["split"], split)
        # several column blocks, degree buckets: two row groups (the halves that go out on two streams), buckets inside each
        assert inf["n_row_groups"] == 2 and inf["reorder"] == 1
        group_row = P.partition_rows(ptr, 2)
        assert np.array_equal(got["group_row"], group_row)
        want = P.plan(ptr, idx, val, inf["seg_len"], True, rb=split[b], re=split[b + 1], skip_empty=0 < b < nb - 1, k4=K // 4,
                      pad=4 * (32 // inf["lanes"]), group_row=group_row)
        want.update(P.light_stream(want, idx, val, 32 // inf["lanes"], inf["light_steps"], k4=K // 4, group_row=group_row))
        want["utask"] = P.unified_tasks(want, want, True, group_row)
        for k in ("row_perm", "light_desc", "ltask", "lpanel", "heavy_rows", "heavy_seg0", "seg_desc", "seg_hrow", "panel", "utask"):
            assert np.array_equal(got[k], want[k]), (b, k)
        # every nonzero of the block lies in its band of B rows
        for r0, beg, d, _ in got["light_desc"][:200]:
            assert np.all((idx[beg:beg + d] >= inf["col_begin"]) & (idx[beg:beg + d] < inf["col_end"]))
        for row, beg, d, _ in got["light_desc"]:
            covered[beg:beg + d] += 1
        # the stream holds every light nonzero exactly once, plus one header per light row
        lp = got["lpanel"]
        assert int((lp[:, 0] >= 0).sum()) == int(got["light_desc"][:, 2].sum())
        assert int(((lp[:, 0] < 0) & (lp[:, 0] != -1)).sum()) == len(got["light_desc"])
        for row, off, ln, nb0 in got["seg_desc"]:
            covered[nb0:nb0 + ln] += 1
    assert np.all(covered == 1)        # the blocks tile A exactly once
    op.close()


@pytest.mark.parametrize("shape,K,nb,seg_len,groups,natural", [("c0", 256, 3, 32, 4, True), ("arxiv", 256, 4, 0, 16, True), ("c0", 32, 3, 16, 1, False),
                                                               ("c0", 128, 1, 64, 0, True), ("c0", 64, 3, 16, 0, False), ("arxiv", 256, 5, 0, 3, False)])
def test_row_group_plan_matches_oracle(shape, K, nb, seg_len, groups, natural):
    """Row groups with column blocks in either row order: tasks cut at group bounds — every array against the numpy
    restatement — and the launches that the row-group halves give (two per pass on two streams with several blocks)."""
    ptr, idx = H.gen_named_graph(shape)
    g, vin, vout = dev_inputs(ptr, idx, K)
    op = H.SpMMB200(g, K, col_blocks=nb, seg_len=seg_len, reorder=0 if natural else 1, row_groups=groups)
    op.preprocess(vin, vout)
    info = op.plan_info(0)
    assert info["n_col_blocks"] == nb
    want_groups = groups or (16 if natural else (2 if nb > 1 else 1))
    assert info["n_row_groups"] == want_groups
    M = g.num_v
    val = g.val.cpu().numpy()
    group_row = P.partition_rows(ptr, want_groups)
    split = P.split_rows(ptr, idx, nb, M) if nb > 1 else np.stack([ptr[:-1], ptr[1:]])
    two_streams = nb > 1 and want_groups > 1        # option split_streams = -1 (auto)
    launches = 0
    for b in range(nb):
        got = op.plan_arrays(b)
        inf = op.plan_info(b)
        if b == 0:
            assert np.array_equal(got["group_row"], group_row)
        want = P.plan(ptr, idx, val, inf["seg_len"], not natural, rb=split[b], re=split[b + 1], skip_empty=0 < b < nb - 1, k4=K // 4,
                      pad=4 * (32 // inf["lanes"]), group_row=group_row)
        want.update(P.light_stream(want, idx, val, 32 // inf["lanes"], inf["light_steps"], k4=K // 4, group_row=group_row))
        want["utask"] = P.unified_tasks(want, want, not natural, group_row)
        for k in ("row_perm", "light_desc", "ltask", "lpanel", "heavy_rows", "heavy_seg0", "seg_desc", "seg_hrow", "panel", "utask"):
            assert np.array_equal(got[k], want[k]), (b, k)
        # the tasks are group-major: the second stream takes the tasks of the second half of the groups
        grp = P.task_groups(want["utask"], want["light_desc"], want["seg_desc"], group_row)
        assert np.all(np.diff(grp) >= 0) and np.all(grp < want_groups)
        n = len(want["utask"])
        cut = int(np.searchsorted(grp, (want_groups + 1) // 2)) if two_streams else n
        launches += (cut > 0) + (n > cut)
    # and it computes the right thing, repeatedly (the segment counters return to zero after every run)
    for _ in range(3):
        vout.fill_(float("nan"))
        op.run(vin, vout)
    torch.cuda.synchronize()
    assert op.launches_per_run == launches
    check_against_oracle(ptr, idx, K, op, g, vin, vout[: M * K].cpu().numpy().reshape(M, K))
    op.close()


def test_unsorted_columns_fall_back_to_one_block():
    rows = [[(5, 1.0), (1, 2.0), (3, 3.0)], [(2, 1.0)], [], [(0, 1.0), (7, -1.0)]] + [[] for _ in range(4)]
    ptr, idx, val = tiny_csr(rows)
    rng = np.random.default_rng(1)
    b = rng.normal(0, 1, (8, 8)).astype(np.float32)
    op, g, vin, vout, got = run_engine(ptr, idx, 8, val=val, b=b, col_blocks=2)
    assert op.plan_info()["n_col_blocks"] == 1
    assert np.array_equal(got.view(np.int32), O.spmm_literal(ptr, idx, val, b, 8).view(np.int32))
    op.close()


def _shuffled_rows(ptr, idx, seed):
    """The same graph with every row's columns in random storage order, and a duplicate column in the longest row."""
    rng = np.random.default_rng(seed)
    idx = idx.copy()
    for r in range(len(ptr) - 1):
        a, b = int(ptr[r]), int(ptr[r + 1])
        idx[a:b] = rng.permutation(idx[a:b])
    r = int(np.argmax(np.diff(ptr)))
    idx[ptr[r]] = idx[ptr[r + 1] - 1]            # the same column twice: stability of the sort is observable
    return idx


@pytest.mark.parametrize("shape,K,opts", [("c0", 64, {"col_blocks": 3, "seg_len": 32}), ("arxiv", 256, {"col_blocks": 4}), ("c0", 33, {})])
def test_column_sorted_operator(shape, K, opts):
    """Rows that are not column-sorted keep ONE column block (bit-exact in storage order); the column-sorted operator
    (spmm_b200_create_column_sorted) gets the bands and equals the oracle run on the stably sorted CSR bit for bit, and the
    oracle run on the original order within the split-row tolerance."""
    ptr, idx0 = H.gen_named_graph(shape)
    idx = _shuffled_rows(ptr, idx0, 7)
    g, vin, vout = dev_inputs(ptr, idx, K)
    M = g.num_v
    src = H.SpMMB200(g, K, **opts)
    src.preprocess(vin, vout)
    assert src.plan_info()["n_col_blocks"] == 1
    op = src.column_sorted(**opts)
    out = torch.full((M * K,), float("nan"), device=DEV)
    op.preprocess(vin, out)
    if "col_blocks" in opts:
        assert op.plan_info()["n_col_blocks"] == opts["col_blocks"]
    op.run(vin, out)
    torch.cuda.synchronize()
    got = out.cpu().numpy().reshape(M, K)
    val = g.val.cpu().numpy()
    # the stable sort, restated: order inside a row by (column, storage position)
    row_of = np.repeat(np.arange(M), np.diff(ptr))
    perm = np.lexsort((np.arange(len(idx)), idx, row_of))
    assert np.array_equal(row_of[perm], row_of)
    check_against_oracle(ptr, idx[perm], K, op, SimpleNamespace(num_v=M, val=torch.from_numpy(val[perm])), vin, got)
    ref0 = O.spmm_f32(ptr, idx, val, vin.cpu().numpy(), K)
    ab = O.spmm_abssum(ptr, idx, val, vin.cpu().numpy(), K)
    assert np.all(np.abs(got.astype(np.float64) - ref0) <= TOL * ab + 1e-30)
    # re-weighted edges reach the sorted copy through refresh_values
    g.val.mul_(-2.0)
    op.refresh_values()
    op.run(vin, out)
    torch.cuda.synchronize()
    heavy = op.heavy_row_set()
    whole = np.asarray([r for r in range(M) if r not in heavy], np.int64)
    want = O.spmm_f32(ptr, idx[perm], val[perm] * np.float32(-2.0), vin.cpu().numpy(), K)
    assert np.array_equal(out.cpu().numpy().reshape(M, K)[whole].view(np.int32), want[whole].view(np.int32))
    op.close()
    src.close()


def test_auto_row_order_rule():
    """Small graphs keep degree buckets; many-wave single-block graphs at K >= 128 use natural order; with column blocks
    (every pass gathers from an L2-resident band whatever the order) buckets again (plan_info reports it)."""
    ptr, idx = H.gen_named_graph("arxiv")
    g, vin, vout = dev_inputs(ptr, idx, 256)
    op = H.SpMMB200(g, 256)
    op.preprocess(vin, vout)
    info = op.plan_info()
    total = int(np.diff(ptr).astype(np.int64).sum()) + g.num_v
    assert info["reorder"] == int(P.auto_reorder(info["lanes"], total, info["resident_warps"])) == 1
    assert P.auto_reorder(32, 126_000_000, info["resident_warps"]) is False
    assert P.auto_reorder(8, 126_000_000, info["resident_warps"]) is True
    op.close()
    op = H.SpMMB200(g, 256, col_blocks=3)
    op.preprocess(vin, vout)
    info = op.plan_info()
    assert info["reorder"] == 1 and info["n_row_groups"] == 2
    vout.fill_(float("nan"))
    op.run(vin, vout)
    torch.cuda.synchronize()
    assert op.launches_per_run == 6          # three passes, each as two launches (row halves) on two streams
    check_against_oracle(ptr, idx, 256, op, g, vin, vout[: g.num_v * 256].cpu().numpy().reshape(g.num_v, 256))
    op.close()


def test_auto_col_blocks_rule():
    assert P.auto_col_blocks(232965, 256, 114615892, 232965) == 5       # reddit K=256: B = 239 MB
    assert P.auto_col_blocks(232965, 32, 114615892, 232965) == 1        # B = 30 MB fits
    assert P.auto_col_blocks(2449029, 256, 123718280, 2449029) == 1     # products: rows too short per block
    assert P.auto_col_blocks(169343, 256, 1166243, 169343) == 1


def test_fill_and_valid_match_oracle():
    for n, seed, stream in [(1, 123, 0), (1000, 123, 1), (1 << 20, 7, 5)]:
        t = H.fill_normal(torch.empty(n, device=DEV), seed, stream)
        assert np.array_equal(t.cpu().numpy(), O.fill_normal(n, seed, stream))
    t = H.fill_normal(torch.empty(4096, device=DEV), 3, 4, mean=1.5, stddev=2.0)
    assert np.array_equal(t.cpu().numpy(), O.fill_normal(4096, 3, 4, 1.5, 2.0))
    a = H.allocate(1000)
    assert a.numel() == 1024                      # data.h:27 rounds up to 512 elements
    rng = np.random.default_rng(0)
    y = rng.normal(0, 1, 100000).astype(np.float32)
    y2 = (y * (1 + rng.normal(0, 0.01, y.size))).astype(np.float32)
    y[:10] = 0
    y2[:5] = 0
    dy, dy2 = torch.from_numpy(y).to(DEV), torch.from_numpy(y2).to(DEV)
    want = O.validate_float(y, y2)
    assert H.valid(dy, dy2, y.size) == want
    if refshim.available():
        # the handout's divide is the fast-math approximate one: allow the 1e-2 boundary cases
        assert abs(refshim.ref_valid(dy, dy2, y.size) - want) <= 3


@pytest.mark.parametrize("shape,K,extra", [("arxiv", 32, {}), ("c0", 64, {"col_blocks": 3}), ("c0", 256, {"col_blocks": 2, "reorder": 0})])
def test_row_partitions_reproduce_full_result(shape, K, extra):
    """SURVEY.md §8e: row blocks balanced by nnz, B replicated; concatenated block results equal the
    single-GPU result bit for bit (per-row arithmetic depends only on the row, seg_len and the column bands)."""
    ptr, idx = H.gen_named_graph(shape)
    opf, g, vin, vout, full = run_engine(ptr, idx, K, seg_len=256, **extra)
    M = g.num_v
    val = g.val
    for parts in (2, 8):
        bounds = H.partition_rows(ptr, parts)
        assert np.array_equal(bounds, P.partition_rows(ptr, parts))
        outs = []
        for r in range(parts):
            r0, r1 = int(bounds[r]), int(bounds[r + 1])
            lptr = H.rebase_ptr(ptr, r0, r1)
            e0, e1 = int(ptr[r0]), int(ptr[r1])
            gl = H.CSR(r1 - r0, e1 - e0, torch.from_numpy(lptr).to(DEV), g.idx[e0:e1].clone(), val[e0:e1].clone())
            o = torch.full((max(1, (r1 - r0) * K),), float("nan"), device=DEV)
            op = H.SpMMB200(gl, K, b_rows=M, seg_len=256, **extra)
            op.preprocess(vin, o)
            assert op.plan_info()["n_col_blocks"] == extra.get("col_blocks", 1)
            op.run(vin, o)
            outs.append(o[: (r1 - r0) * K].cpu().numpy())
            op.close()
        cat = np.concatenate(outs).reshape(M, K)
        assert np.array_equal(cat.view(np.int32), full.view(np.int32))
    opf.close()


# ---- BASELINE full sizes: size-independent properties ---------------------------------------------------

def _full_size_properties(shape, K):
    ptr, idx = H.gen_named_graph(shape)
    op, g, vin, vout, _ = run_engine(ptr, idx, K)
    M, nnz = g.num_v, g.num_e
    C1 = vout[: M * K].view(M, K)
    # (a) sampled row ranges against the oracle (bit-exact when whole, tolerance when split)
    val_h, b_h = g.val.cpu().numpy(), vin.cpu().numpy()
    deg = np.diff(ptr)
    heavy = op.heavy_row_set()
    picks = [0, M // 3, M - 64, int(np.argmax(deg)) - 3]
    for r0 in picks:
        r0 = max(0, min(M - 64, r0))
        ref = O.spmm_f32(ptr, idx, val_h, b_h, K, row_begin=r0, row_end=r0 + 64)[r0:r0 + 64]
        got = C1[r0:r0 + 64].cpu().numpy()
        for i in range(64):
            if (r0 + i) in heavy:
                scale = np.abs(b_h.reshape(M, K)[idx[ptr[r0 + i]:ptr[r0 + i + 1]]] * val_h[ptr[r0 + i]:ptr[r0 + i + 1], None]).sum(0)
                assert np.all(np.abs(got[i].astype(np.float64) - ref[i]) <= TOL * scale + 1e-30)
            else:
                assert np.array_equal(got[i].view(np.int32), ref[i].view(np.int32)), r0 + i
    # (b) checksum of checksums: sum_r C[r,:] == sum_c (sum of column c's values) * B[c,:]   (fp64)
    colw = torch.zeros(M, dtype=torch.float64, device=DEV)
    colw.index_add_(0, g.idx.long(), g.val.double())
    want = (colw[:, None] * vin.view(M, K).double()).sum(0)
    got = C1.double().sum(0)
    scale = (colw.abs()[:, None] * vin.view(M, K).double().abs()).sum(0)
    assert torch.all((got - want).abs() <= 1e-6 * scale)
    # (c) linearity in B: A(2*B) == 2*A(B) exactly (scaling by 2 commutes with rounding)
    vin2 = vin * 2
    vout2 = torch.empty_like(vout)
    op.run(vin2, vout2)
    assert torch.equal(vout2[: M * K], vout[: M * K] * 2)
    # (d) idempotence
    op.run(vin, vout2)
    assert torch.equal(vout2[: M * K], vout[: M * K])
    # (e) the reference's criterion against itself is clean (no NaN/Inf produced)
    assert torch.isfinite(C1).all()
    op.close()


def test_reddit_k256_full_size_properties():
    _full_size_properties("reddit", 256)


def test_products_k256_full_size_properties():
    _full_size_properties("products", 256)


def _abs_sum_device(g, vin, M, K, chunk=1 << 20):
    """sum_i |B[idx_i, j] * val_i| per output element, on the device, in nnz chunks (the tolerance scale)."""
    deg = (g.ptr[1: M + 1] - g.ptr[:M]).long()
    rows = torch.repeat_interleave(torch.arange(M, device=DEV), deg)
    ab = torch.zeros(M, K, device=DEV)
    b = vin.view(-1, K)
    for e0 in range(0, g.num_e, chunk):
        e1 = min(g.num_e, e0 + chunk)
        ab.index_add_(0, rows[e0:e1], (b[g.idx[e0:e1].long()] * g.val[e0:e1, None]).abs_())
    return ab


@pytest.mark.parametrize("shape", ["reddit", "products"])
def test_full_output_against_reference_kernel_k256(shape, golden_dir):
    """BASELINE configs 3-4, ALL M*K elements (the reference validates every element: test_spmm.cu:31-44): the engine
    against spmm_kernel_ref's output on identical device inputs — whole rows bit-equal, split rows within
    1e-5 * sum|terms|, and the reference's own criterion. No sampling."""
    K = 256
    ptr, idx = H.gen_named_graph(shape)
    g, vin, vout = dev_inputs(ptr, idx, K)
    M = g.num_v
    op = H.SpMMB200(g, K)
    op.preprocess(vin, vout)
    op.run(vin, vout)
    ref_h = reference_output(golden_dir, f"{shape}_k{K}", ptr, idx, K, g, vin)
    ref_out = torch.from_numpy(ref_h.ravel()).to(DEV)
    torch.cuda.synchronize()
    got, ref = vout[: M * K].view(M, K), ref_out.view(M, K)
    whole = torch.ones(M, dtype=torch.bool, device=DEV)
    heavy = sorted(op.heavy_row_set())
    if heavy:
        whole[torch.tensor(heavy, device=DEV)] = False
    assert int(whole.sum()) + len(heavy) == M
    assert torch.equal(got[whole].view(torch.int32), ref[whole].view(torch.int32)), "whole rows must be bit-exact"
    ab = _abs_sum_device(g, vin, M, K)
    err = (got.double() - ref.double()).abs()
    assert bool((err <= TOL * ab.double() + 1e-30).all()), float((err / (ab.double() + 1e-30)).max())
    assert O.validate_float(got.cpu().numpy(), ref_h) < M * K // 10000 + 1
    if refshim.available():
        assert refshim.ref_valid(vout, ref_out, M * K) < M * K // 10000 + 1
    info = op.plan_info()
    print(f"{shape} K={K}: {M - len(heavy)} whole rows bit-equal, {len(heavy)} split rows max rel "
          f"{float((err / (ab.double() + 1e-30)).max()):.2e}, col_blocks={info['n_col_blocks']}")
    op.close()


def test_host_bands_layout_for_run_host():
    """Option host_bands: the last column block is the last 40 % of B (its pass is bound by the PCIe transfer of C), the
    blocks before it share the rest. Bounds and row splits against the oracle; result unchanged; run_host bit-equal."""
    ptr, idx = H.gen_named_graph("c0")
    K, nb = 64, 4
    op, g, vin, vout, got = run_engine(ptr, idx, K, col_blocks=nb, host_bands=1, seg_len=32)
    M = g.num_v
    bounds = P.host_band_bounds(nb, M)
    assert bounds == [0, 819, 1638, 2457, 4096]
    info = op.plan_info()
    assert info["n_col_blocks"] == nb
    split = P.split_rows(ptr, idx, nb, M, bounds=bounds)
    for b in range(nb):
        inf = op.plan_info(b)
        assert (inf["col_begin"], inf["col_end"]) == (bounds[b], bounds[b + 1])
    assert np.array_equal(op.plan_arrays(0)["split"], split)
    check_against_oracle(ptr, idx, K, op, g, vin, got)
    h_in, h_out = vin.cpu().pin_memory(), torch.full((M * K,), float("nan")).pin_memory()
    for _ in range(2):
        op.run_host(h_in, h_out)
        assert np.array_equal(h_out.numpy().view(np.int32), got.ravel().view(np.int32))
    op.close()


def test_refresh_values_after_in_place_update():
    """The plan snapshots idx/val into its panels (spmm_b200.h: SNAPSHOT); refresh_values re-stages them without a new
    plan. The reference's SpMMOpt::run reads idx/val live (PA4/workspace/src/spmm_opt.cu:22-25)."""
    ptr, idx = H.gen_named_graph("c0")
    for K, opts in ((32, {"seg_len": 64}), (256, {"col_blocks": 3, "seg_len": 32}), (33, {})):
        g, vin, vout = dev_inputs(ptr, idx, K)
        op = H.SpMMB200(g, K, **opts)
        op.preprocess(vin, vout)
        op.run(vin, vout)
        g.val.mul_(-3.0)                       # edge re-weighting in place
        op.refresh_values()
        op.run(vin, vout)
        torch.cuda.synchronize()
        got = vout[: g.num_v * K].cpu().numpy().reshape(g.num_v, K)
        check_against_oracle(ptr, idx, K, op, g, vin, got)
        op.close()


def test_b_rows_change_invalidates_plan_and_bands_stay_inside_b():
    ptr, idx = H.gen_named_graph("c0")
    K = 32
    g, vin, vout = dev_inputs(ptr, idx, K)
    op = H.SpMMB200(g, K)
    op.preprocess(vin, vout)
    op.set_option("b_rows", g.num_v + 8)
    with pytest.raises(H.SpmmB200Error) as e:
        op.run(vin, vout)
    assert e.value.code == -2
    op.close()
    # 10 rows of B, 7 requested bands: ceil(10/7) = 2 rows per band -> 5 bands, none outside B
    ptr2 = np.arange(0, 11, dtype=np.int32) * 3
    idx2 = np.tile(np.array([0, 4, 9], np.int32), 10)
    op, g2, vin2, vout2, got = run_engine(ptr2, idx2, 8, col_blocks=7)
    for b in range(op.plan_info()["n_col_blocks"]):
        info = op.plan_info(b)
        assert 0 <= info["col_begin"] < info["col_end"] <= 10
    assert op.plan_info()["n_col_blocks"] == 5
    check_against_oracle(ptr2, idx2, 8, op, g2, vin2, got)
    h_in, h_out = vin2.cpu().pin_memory(), torch.empty(80).pin_memory()
    op.run_host(h_in, h_out)
    assert np.array_equal(h_out.numpy().reshape(10, 8).view(np.int32), got.view(np.int32))
    op.close()


def test_feat_zero_is_a_no_op():
    ptr, idx = H.gen_named_graph("c0")
    g, vin, vout = dev_inputs(ptr, idx, 4)
    op = H.SpMMB200(g, 0)
    op.preprocess(vin, vout)
    op.run(vin, vout)
    op.set_feat(4)
    op.preprocess(vin, vout)
    op.run(vin, vout)
    torch.cuda.synchronize()
    check_against_oracle(ptr, idx, 4, op, g, vin, vout[: g.num_v * 4].cpu().numpy().reshape(-1, 4))
    op.close()


# ---- the transposed operator: dB = A^T dC (SURVEY.md 8f-3; no reference counterpart, parity unpinned) ---------

@pytest.mark.parametrize("shape,K,opts", [("c0", 32, {}), ("c0", 256, {"seg_len": 32}), ("arxiv", 256, {}), ("arxiv", 32, {}),
                                           ("c0", 33, {}), pytest.param("c0", 64, {"col_blocks": 3}, id="c0-64-col_blocks3")])
def test_transposed_operator_matches_oracle(shape, K, opts):
    ptr, idx = H.gen_named_graph(shape)
    g, vin, vout = dev_inputs(ptr, idx, K)
    M = g.num_v
    fwd = H.SpMMB200(g, K)
    bwd = fwd.transposed(**opts)
    dc = H.fill_normal(torch.empty(M * K, device=DEV), 77, 3)
    db = torch.full((M * K,), float("nan"), device=DEV)
    bwd.preprocess(dc, db)
    bwd.run(dc, db)
    torch.cuda.synchronize()
    got = db.cpu().numpy().reshape(M, K)
    want, ab = O.spmm_t_f32(ptr, idx, g.val.cpu().numpy(), dc.cpu().numpy(), K, with_abs=True)
    heavy = bwd.heavy_row_set()
    whole = np.asarray([r for r in range(M) if r not in heavy], np.int64)
    assert np.array_equal(got[whole].view(np.int32), want[whole].view(np.int32)), "whole rows of A^T must be bit-exact"
    assert np.all(np.abs(got.astype(np.float64) - want) <= TOL * ab + 1e-30)
    # adjoint identity in fp64: <A x, y> == <x, A^T y>
    fwd.preprocess(vin, vout)
    fwd.run(vin, vout)
    lhs = float((vout[: M * K].double() * dc.double()).sum())
    rhs = float((vin[: M * K].double() * db.double()).sum())
    assert abs(lhs - rhs) <= 1e-6 * float((vout[: M * K].double().abs() * dc.double().abs()).sum())
    # edge re-weighting: the transposed operator re-reads the source operator's values
    g.val.mul_(0.5)
    bwd.refresh_values()
    bwd.run(dc, db)
    torch.cuda.synchronize()
    assert np.array_equal(db.cpu().numpy().reshape(M, K)[whole].view(np.int32), (want[whole] * np.float32(0.5)).view(np.int32))
    bwd.close()
    fwd.close()


def test_transposed_operator_of_a_row_block():
    """A row block of a larger graph (b_rows > num_v): A^T has b_rows rows and gathers from the block's rows of dC."""
    ptr, idx = H.gen_named_graph("c0")
    K, M = 32, len(ptr) - 1
    bounds = H.partition_rows(ptr, 3)
    val = O.fill_normal(len(idx), 123, 1)
    total = np.zeros((M, K), np.float64)
    dc_full = O.fill_normal(M * K, 9, 4).reshape(M, K)
    for part in range(3):
        r0, r1 = int(bounds[part]), int(bounds[part + 1])
        lptr = H.rebase_ptr(ptr, r0, r1)
        e0, e1 = int(ptr[r0]), int(ptr[r1])
        g, _, _ = dev_inputs(lptr, idx[e0:e1], K, val=val[e0:e1], b_rows=M)
        fwd = H.SpMMB200(g, K, b_rows=M)
        bwd = fwd.transposed()
        assert (bwd.num_v, bwd.b_rows) == (M, r1 - r0)
        dc = torch.from_numpy(dc_full[r0:r1].ravel().copy()).to(DEV)
        db = torch.empty(M * K, device=DEV)
        bwd.preprocess(dc, db)
        bwd.run(dc, db)
        torch.cuda.synchronize()
        want = O.spmm_t_f32(lptr, idx[e0:e1], val[e0:e1], dc_full[r0:r1].ravel(), K, b_rows=M)
        heavy = bwd.heavy_row_set()
        whole = np.asarray([r for r in range(M) if r not in heavy], np.int64)
        assert np.array_equal(db.cpu().numpy().reshape(M, K)[whole].view(np.int32), want[whole].view(np.int32))
        total += db.cpu().numpy().reshape(M, K)
        bwd.close()
        fwd.close()
    full = O.spmm_t_f32(ptr, idx, val, dc_full.ravel(), K)
    assert np.allclose(total, full, rtol=1e-4, atol=1e-5)     # the blocks' gradients add up to the whole graph's


# ---- multi-GPU driver behind the C ABI (spmm_b200_mg_*) -----------------------------------------------------

def _mg_devices():
    n = torch.cuda.device_count()
    cases = [[0], [0, 0, 0]]            # one box GPU listed three times exercises partition, push and gather logic
    if n >= 2:
        cases.append(list(range(min(n, 8))))
    return cases


@pytest.mark.parametrize("shape,K", [("c0", 32), ("arxiv", 256)])
def test_mg_run_host_and_stacked_layers(shape, K):
    ptr, idx = H.gen_named_graph(shape)
    M, nnz = len(ptr) - 1, len(idx)
    val = O.fill_normal(nnz, 123, 1)
    b = O.fill_normal(M * K, 123, 2)
    g, vin, vout = dev_inputs(ptr, idx, K, val=val, b=b)
    op = H.SpMMB200(g, K)
    op.preprocess(vin, vout)
    op.run(vin, vout)
    vout2 = torch.empty_like(vout)
    op.run(vout, vout2)                                  # second stacked layer on one GPU
    torch.cuda.synchronize()
    want1, want2 = vout[: M * K].cpu(), vout2[: M * K].cpu()
    op.close()
    for devs in _mg_devices():
        mg = H.MultiGpuSpMM(ptr, idx, val, K, devices=devs)
        info = mg.info()
        assert info["n_devices"] == len(devs) and info["bounds"][0] == 0 and info["bounds"][-1] == M
        assert np.array_equal(info["bounds"], H.partition_rows(ptr, len(devs)))
        mg.preprocess()
        h_in = torch.from_numpy(b).pin_memory()
        h_out = torch.full((M * K,), float("nan")).pin_memory()
        for _ in range(2):                               # twice: the second call orders its pushes after the first's passes
            mg.run_host(h_in, h_out)
        assert torch.equal(h_out.view(torch.int32), want1.view(torch.int32)), devs
        # stacked layers, device-resident: NCCL (or copy) all-gather-v vs the fused epilogue — bit-identical
        for fused in (False, True):
            mg.set_fused(fused)
            mg.run_host(h_in, h_out)                     # B = input on every device again
            mg.run()
            if not fused:
                mg.allgather()
            mg.sync()
            mg.swap()                                    # layer 1's C is layer 2's B
            mg.run()
            if not fused:
                mg.allgather()
            mg.sync()
            for gdev in range(len(devs)):
                bufs = mg.device_buffers(gdev)
                full = torch.empty(M * K, device=f"cuda:{devs[gdev]}")
                _copy_from_ptr(full, bufs["c_full"], devs[gdev])
                assert torch.equal(full.cpu().view(torch.int32), want2.view(torch.int32)), (devs, fused, gdev)
            mg.swap()
        mg.close()


def _copy_from_ptr(dst, src_ptr, device):
    """device-to-device copy from a raw pointer (the mg driver's buffers are not torch tensors)."""
    import ctypes as C
    rt = C.CDLL("libcudart.so.12")
    with torch.cuda.device(device):
        torch.cuda.synchronize()
        rc = rt.cudaMemcpy(C.c_void_p(dst.data_ptr()), C.c_void_p(src_ptr), C.c_size_t(dst.numel() * 4), 3)
        assert rc == 0, rc


# ---- the reference's test driver, restated without gtest (tests/cpp/unit_tests.cpp) ---------------------

def test_cpp_harness_validation_and_timing(tmp_path):
    import subprocess
    from conftest import ROOT
    exe = os.path.join(ROOT, "tests", "cpp", "unit_tests")
    if not os.path.exists(exe):
        subprocess.run(["make", "-C", os.path.join(ROOT, "tests", "cpp")], check=True, capture_output=True)
    # synthetic shape
    r = subprocess.run([exe, "--shape", "arxiv", "--len", "32"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "[  PASSED  ] 2 tests." in r.stdout
    assert "time = " in r.stderr and "(double)" in r.stderr          # the line PA4/workspace/plot.py:13-27 parses
    # reference file format: --dataset/--datadir, as run_all.sh:11 calls it
    ptr, idx = H.gen_named_graph("c0")
    H.write_graph(str(tmp_path), "c0", ptr, idx, text=True)
    r = subprocess.run([exe, "--dataset", "c0", "--datadir", str(tmp_path), "--len", "256"], capture_output=True,
                       text=True, timeout=300)
    assert r.returncode == 0 and "[  PASSED  ] 2 tests." in r.stdout, r.stdout + r.stderr


def test_run_all_sweep_subset(tmp_path):
    """run_all.sh restated: a subset of the 13 dataset shapes through the harness, log parsable like plot.py does."""
    import re
    import subprocess
    from conftest import ROOT
    log = str(tmp_path / "out.log")
    r = subprocess.run([os.path.join(ROOT, "tests", "cpp", "run_all.py"), "--len", "32", "--log", log, "collab", "ddi", "am"],   # ddi at K=32: every row is heavy
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    text = open(log).read()
    # plot.py:13-27: dataset from `dset = "name"`, times from `time = x (double)`
    assert re.findall(r'dset = "([a-z_.0-9]+)"', text) == ["collab", "ddi", "am"]
    assert len(re.findall(r"time = ([0-9.e+-]+) \(double\)", text)) == 3
    assert text.count("[  PASSED  ] 2 tests.") == 3


@pytest.mark.parametrize("shape,K,opts", [("c0", 32, {}), ("arxiv", 256, {}), ("c0", 256, {"col_blocks": 3, "seg_len": 32})])
def test_stacked_layer_epilogue_local_targets(shape, K, opts):
    """spmm_b200_set_gather with local buffers standing in for peers: every finished row lands at its offset in
    every target, bit-equal to vout; rows outside this handle's block stay untouched."""
    ptr, idx = H.gen_named_graph(shape)
    g, vin, vout = dev_inputs(ptr, idx, K)
    M = g.num_v
    pad = 5
    targets = [torch.full(((M + 2 * pad) * K,), -7.0, device=DEV) for _ in range(3)]
    op = H.SpMMB200(g, K, **opts)
    op.set_gather(targets, row_offset=pad)
    op.preprocess(vin, vout)
    op.run(vin, vout)
    torch.cuda.synchronize()
    for t in targets:
        assert torch.equal(t[pad * K:(pad + M) * K], vout[: M * K])
        assert bool((t[: pad * K] == -7.0).all()) and bool((t[(pad + M) * K:] == -7.0).all())
    check_against_oracle(ptr, idx, K, op, g, vin, vout[: M * K].cpu().numpy().reshape(M, K))
    # off again: targets no longer written
    op.set_gather([], 0)
    op.preprocess(vin, vout)
    for t in targets:
        t.fill_(1.0)
    op.run(vin, vout)
    torch.cuda.synchronize()
    assert all(bool((t == 1.0).all()) for t in targets)
    op.close()


# ---- the reference's own, unmodified test driver with the engine dropped in (INTEGRATION.md §2) ----------

_DROPIN = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle", "_ref", "unit_tests_dropin")


@pytest.mark.skipif(not os.path.exists(_DROPIN), reason="oracle/_ref/unit_tests_dropin not built (needs /root/reference at build time)")
@pytest.mark.parametrize("shape,K", [("c0", 32), ("arxiv", 32), ("arxiv", 256), ("ddi", 256)])
def test_reference_test_driver_with_engine_dropped_in(tmp_path, shape, K):
    """PA4/handout/test/main.cpp + test_spmm.cu, compiled unmodified with tests/cpp/dropin/spmm_opt.h in place of the
    handout's: SpMMTest.validation compares the engine with the reference's SpMMRef kernel on cuRAND inputs and applies
    the reference's valid(); cusparse_performance / opt_performance time cuSPARSE and the engine the reference's way."""
    import re
    import subprocess
    ptr, idx = H.gen_named_graph(shape)
    H.write_graph(str(tmp_path), shape, ptr, idx, text=False)     # the reference's binary dump format
    r = subprocess.run([_DROPIN, "--dataset", shape, "--datadir", str(tmp_path), "--len", str(K)], capture_output=True,
                       text=True, timeout=600)
    out = r.stdout + r.stderr
    assert r.returncode == 0, out[-3000:]
    assert "[       OK ] SpMMTest.validation" in out and "[  PASSED  ] 3 tests." in out, out[-3000:]
    times = [float(x) for x in re.findall(r"time = ([0-9.e+-]+) \(double\)", out)]
    assert len(times) == 2 and all(t > 0 for t in times)          # cuSPARSE, then the engine (test_spmm.cu:46-62)


@pytest.mark.parametrize("K,opts", [(32, {}), (64, {"col_blocks": 3})])
def test_run_is_capturable_in_a_cuda_graph(K, opts):
    """run() makes no host synchronisation, so a launch-bound caller can capture it once and replay it — also when the
    passes go out on two streams (fork / join inside the capture)."""
    ptr, idx = H.gen_named_graph("arxiv")
    g, vin, vout = dev_inputs(ptr, idx, K)
    op = H.SpMMB200(g, K, **opts)
    op.preprocess(vin, vout)
    op.run(vin, vout)
    torch.cuda.synchronize()
    want = vout.clone()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(s):
        op.run(vin, vout)                      # warm-up on the capture stream
        s.synchronize()
        with torch.cuda.graph(graph, stream=s):
            op.run(vin, vout)
    for _ in range(3):
        vout.fill_(float("nan"))
        graph.replay()
        torch.cuda.synchronize()
        assert torch.equal(vout, want)
    op.close()


def test_fuzz_random_graphs_and_options():
    """Seeded sweep over small random graphs x K x plan options: every combination must satisfy the parity bar."""
    rng = np.random.default_rng(2024)
    for case in range(48):
        m = int(rng.integers(1, 1500))
        mean = float(rng.choice([0.5, 3, 20, 120]))
        deg = np.minimum(rng.poisson(mean, m) * (rng.random(m) < 0.8) + (rng.random(m) < 0.02) * rng.integers(0, m + 1, m), m).astype(np.int64)
        ptr = np.zeros(m + 1, np.int32)
        np.cumsum(deg, out=ptr[1:])
        idx = np.concatenate([np.sort(rng.choice(m, int(d), replace=False)) for d in deg] + [np.zeros(0, np.int64)]).astype(np.int32)
        K = int(rng.choice([4, 8, 12, 32, 36, 64, 128, 256, 260, 512, 5, 33]))
        opts = {}
        if K % 4 == 0:
            if rng.random() < 0.6:
                opts["seg_len"] = int(rng.choice([1, 2, 7, 16, 64, 300]))
            if rng.random() < 0.4:
                opts["col_blocks"] = int(rng.integers(1, 7))
            if rng.random() < 0.4:
                opts["light_steps"] = int(rng.choice([1, 2, 5, 16, 100]))
            if rng.random() < 0.3:
                opts["kslice"] = int(rng.choice([4, 16, 32, 64, 128]))
            if rng.random() < 0.3:
                opts["tune"] = 1
            if rng.random() < 0.3:
                opts["block"] = int(rng.choice([32, 64, 256]))
        if rng.random() < 0.4:
            opts["reorder"] = int(rng.integers(0, 2))
        op, g, vin, vout, got = run_engine(ptr, idx, K, **opts)
        try:
            check_against_oracle(ptr, idx, K, op, g, vin, got)
        except AssertionError as e:
            raise AssertionError(f"fuzz case {case}: m={m} nnz={len(idx)} K={K} opts={opts}: {e}")
        finally:
            op.close()


@pytest.mark.parametrize("workload", ["c0_k32", "reddit_k256"])
def test_bench_dump_outputs(tmp_path, workload):
    """bench.py --dump-outputs: C of the last timed step on the benchmark's seeded inputs, against the oracle — the whole
    of C (c0, K=32), and the seeded sample of rows when C exceeds bench.DUMP_BYTES (reddit, K=256: 238 MB)."""
    import subprocess
    import sys
    from conftest import ROOT
    import bench
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", workload, "--steps", "2", "--no-also",
                        "--no-cpu-baseline", "--sustain-seconds", "0.05", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == 2
    c, rows = np.load(tmp_path / "C.npy"), np.load(tmp_path / "C_rows.npy")
    shape, K = bench.WORKLOADS[workload]
    ptr, idx = H.gen_named_graph(shape)
    M = len(ptr) - 1
    n = min(M, bench.DUMP_BYTES // (4 * K + 8))
    assert c.dtype == np.float32 and rows.dtype == np.float64 and c.shape == (n, K) and rows.shape == (n,)
    assert c.nbytes + rows.nbytes <= bench.DUMP_BYTES
    want_rows = np.arange(M) if n == M else np.sort(np.random.default_rng(bench.SEED).choice(M, n, replace=False))
    assert np.array_equal(rows, want_rows.astype(np.float64))
    val, b = O.fill_normal(len(idx), bench.SEED, 1), O.fill_normal(M * K, bench.SEED, 2)
    ref, ab = O.spmm_f32(ptr, idx, val, b, K)[want_rows], O.spmm_abssum(ptr, idx, val, b, K)[want_rows]
    assert np.all(np.abs(c.astype(np.float64) - ref) <= TOL * ab + 1e-30)


def test_plain_c_example_runs(tmp_path):
    """examples/minimal.c end to end: plain C host, CUDA runtime API, the C ABI — prints and checks a 3x3 product."""
    import subprocess
    from conftest import ROOT
    cuda = "/usr/local/cuda"
    exe = str(tmp_path / "minimal")
    r = subprocess.run(["gcc", "-std=c99", "-I", os.path.join(ROOT, "include"), "-I", os.path.join(cuda, "include"),
                        os.path.join(ROOT, "examples", "minimal.c"), "-L", os.path.join(ROOT, "hpc_b200"), "-lspmm_b200",
                        "-L", os.path.join(cuda, "lib64"), "-lcudart", "-Wl,-rpath," + os.path.join(ROOT, "hpc_b200"), "-o", exe],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stdout + r.stderr
    assert [float(x) for x in r.stdout.split()] == [32, 37, 42, 47, 0, 0, 0, 0, 0, -1, -2, -3]


def test_cpp_multi_gpu_example_runs(tmp_path):
    """examples/multi_gpu.cpp: the spmm_b200_mg_* driver from a C++ host — host-buffer call and two stacked layers (NCCL
    all-gather-v vs the kernel epilogue), on every visible GPU and with one GPU listed three times."""
    import subprocess
    from conftest import ROOT
    cuda = "/usr/local/cuda"
    exe = str(tmp_path / "multi_gpu")
    r = subprocess.run(["g++", "-std=c++17", "-I", os.path.join(ROOT, "include"), "-I", os.path.join(cuda, "include"),
                        os.path.join(ROOT, "examples", "multi_gpu.cpp"), "-L", os.path.join(ROOT, "hpc_b200"), "-lspmm_b200",
                        "-L", os.path.join(cuda, "lib64"), "-lcudart", "-Wl,-rpath," + os.path.join(ROOT, "hpc_b200"), "-o", exe],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    for n in sorted({1, 3, torch.cuda.device_count()}):
        r = subprocess.run([exe, str(n)], capture_output=True, text=True, timeout=300)
        assert r.returncode == 0, (n, r.stdout + r.stderr)
        assert r.stdout.count("ok") == 2, r.stdout
