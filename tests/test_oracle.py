"""The CPU oracle (oracle/spmm_oracle.c) against hand-checkable cases, its own literal form,
and the committed golden vectors. The reference ships no SpMM golden vector (SURVEY.md §8c);
tests/test_gpu_parity.py pins this oracle bit-for-bit against the reference kernel's stored
outputs (tests/golden/make_reference_golden.py)."""
import json
import os

import numpy as np
import pytest

from conftest import tiny_csr
from oracle import cpu as O


def test_hand_checked_tiny():
    # 3x3: row0 = 2*B[1] + 3*B[2]; row1 empty; row2 = -1*B[0]
    ptr, idx, val = tiny_csr([[(1, 2.0), (2, 3.0)], [], [(0, -1.0)]])
    b = np.arange(12, dtype=np.float32).reshape(3, 4)
    out = O.spmm_literal(ptr, idx, val, b, 4)
    want = np.stack([2 * b[1] + 3 * b[2], np.zeros(4, np.float32), -b[0]])
    assert np.array_equal(out, want)
    assert np.array_equal(O.spmm_f32(ptr, idx, val, b, 4), want)


def test_duplicate_columns_accumulate_in_order():
    # spmm_ref.cu:11-14 does not deduplicate: both entries contribute, in CSR order
    ptr, idx, val = tiny_csr([[(0, 1e8), (0, 1.0), (0, -1e8)]])
    b = np.ones((1, 1), np.float32)
    assert O.spmm_literal(ptr, idx, val, b, 1)[0, 0] == np.float32(0.0)   # 1e8 + 1 rounds to 1e8 in fp32
    ptr, idx, val = tiny_csr([[(0, 1e8), (0, -1e8), (0, 1.0)]])
    assert O.spmm_literal(ptr, idx, val, b, 1)[0, 0] == np.float32(1.0)


def test_fma_is_single_rounding():
    # a*b + c with one rounding differs from round(a*b) + c
    a = np.float32(1 + 2 ** -12)
    ptr, idx, val = tiny_csr([[(0, -1.0), (1, a)]])
    b = np.asarray([[np.float32(a * a)], [a]], np.float32)   # row0 = -fl(a*a) + a*a (exact inside fma)
    out = O.spmm_literal(ptr, idx, val, b, 1)[0, 0]
    assert out == np.float32(2.0 ** -24) * 0 + np.float32(float(a) * float(a) - float(np.float32(a * a)))


@pytest.mark.parametrize("feat", [1, 3, 32, 100])
def test_interchanged_equals_literal(feat):
    rng = np.random.default_rng(feat)
    m = 300
    deg = rng.integers(0, 40, m)
    deg[7] = 257
    ptr = np.zeros(m + 1, np.int32)
    np.cumsum(deg, out=ptr[1:])
    idx = rng.integers(0, m, ptr[-1]).astype(np.int32)
    val = rng.normal(0, 0.1, ptr[-1]).astype(np.float32)
    b = rng.normal(0, 0.1, (m, feat)).astype(np.float32)
    lit = O.spmm_literal(ptr, idx, val, b, feat)
    for nt in (1, 4):
        assert np.array_equal(lit.view(np.int32), O.spmm_f32(ptr, idx, val, b, feat, nthreads=nt).view(np.int32))
    # row range + ftz variants agree on normal-range data
    part = O.spmm_f32(ptr, idx, val, b, feat, row_begin=10, row_end=20)
    assert np.array_equal(part[10:20], lit[10:20]) and not part[:10].any() and not part[20:].any()
    assert np.array_equal(O.spmm_f32(ptr, idx, val, b, feat, ftz=True), lit)
    # fp64 agrees to fp32 accuracy
    f64 = O.spmm_f64(ptr, idx, val, b, feat)
    ab = O.spmm_abssum(ptr, idx, val, b, feat)
    assert np.all(np.abs(lit - f64) <= 1e-5 * ab + 1e-30)


def test_ftz_model():
    tiny = np.float32(1e-40)   # subnormal
    ptr, idx, val = tiny_csr([[(0, 1.0)]])
    b = np.asarray([[tiny]], np.float32)
    assert O.spmm_literal(ptr, idx, val, b, 1, ftz=False)[0, 0] == tiny
    assert O.spmm_literal(ptr, idx, val, b, 1, ftz=True)[0, 0] == 0.0


def test_validate_float_semantics():
    # valid.cu:8: |(ref-ans)/ref| > 1e-2; first argument normalises; 0/0 not counted, x/0 counted
    ref = np.asarray([1.0, 1.0, 0.0, 0.0, 100.0, -2.0], np.float32)
    ans = np.asarray([1.005, 1.02, 0.0, 1e-9, 98.9, -2.0], np.float32)
    assert O.validate_float(ref, ans) == 3
    assert O.validate_int(np.arange(5), np.asarray([0, 1, 9, 3, 9])) == 2


def test_fill_normal_moments_and_streams():
    x = O.fill_normal(1 << 20, 123, 0)
    assert abs(float(x.mean())) < 5e-4 and abs(float(x.std()) - 0.1) < 5e-4
    assert float(np.abs(x).max()) < 0.5      # Irwin-Hall support is +-4.9 sigma
    y = O.fill_normal(1 << 10, 123, 1)
    assert not np.array_equal(x[:1 << 10], y)
    assert np.array_equal(O.fill_normal(1000, 123, 0), x[:1000])      # counter-based: prefix-stable
    z = O.fill_normal(1000, 5, 7, mean=2.0, stddev=0.5)
    assert abs(float(z.mean()) - 2.0) < 0.1


def test_fill_normal_numpy_restatement():
    """Independent numpy restatement of oracle_fill_normal's published definition."""
    from oracle.graph_oracle import mix64
    n, seed, stream = 4097, 123, 2
    with np.errstate(over="ignore"):
        key = mix64(np.uint64(seed) ^ mix64(np.uint64(stream) * np.uint64(0x632BE59BD9B4E019) + np.uint64(0x1234567)))
        i = np.arange(n, dtype=np.uint64)
        a, b = mix64(key + np.uint64(2) * i), mix64(key + np.uint64(2) * i + np.uint64(1))
    s16 = lambda v: sum(((v >> np.uint64(sh)) & np.uint64(0xFFFF)).astype(np.int64) for sh in (0, 16, 32, 48))
    t = (s16(a) + s16(b) - 262140).astype(np.float32)
    want = t * np.float32(0.1 / 53510.0) + np.float32(0.0)
    assert np.array_equal(want.astype(np.float32), O.fill_normal(n, seed, stream))


def test_student_task_split():
    # PA4/workspace/src/spmm_opt.cu:43-54
    ptr = np.asarray([0, 0, 256, 513, 1300], np.int32)
    t = O.student_tasks(ptr)
    want = [(1, 0, 256), (2, 256, 512), (2, 512, 513), (3, 513, 769), (3, 769, 1025), (3, 1025, 1281), (3, 1281, 1300)]
    assert t.tolist() == [list(w) for w in want]


def test_golden_vectors(golden_dir):
    """Committed fixtures (tests/golden/make_golden.py): inputs regenerate from seeds, outputs are stored."""
    meta = json.load(open(os.path.join(golden_dir, "golden.json")))
    data = np.load(os.path.join(golden_dir, "golden.npz"))
    for case in meta["cases"]:
        n = case["name"]
        ptr, idx = data[f"{n}_ptr"], data[f"{n}_idx"]
        val = O.fill_normal(len(idx), case["seed"], 1)
        b = O.fill_normal((len(ptr) - 1) * case["K"], case["seed"], 2)
        out = O.spmm_f32(ptr, idx, val, b, case["K"])
        assert np.array_equal(out.view(np.int32), data[f"{n}_out"].view(np.int32).reshape(out.shape)), n


def test_transposed_product_oracle_is_the_forward_oracle_on_the_transposed_csr():
    """oracle_spmm_t_f32 (dB = A^T dC, chains in CSR storage order) == the forward restatement run on A^T built by
    scipy with each row's entries by ascending row of A — bitwise; and the fp64 abs-sum agrees."""
    import scipy.sparse as sp
    import hpc_b200 as H
    ptr, idx = H.gen_named_graph("c0")
    M, nnz, K = len(ptr) - 1, len(idx), 8
    val = O.fill_normal(nnz, 5, 1)
    dc = O.fill_normal(M * K, 5, 2)
    got, ab = O.spmm_t_f32(ptr, idx, val, dc, K, with_abs=True)
    # A^T with explicit positions so that values follow the permutation exactly
    at = sp.csr_matrix((np.arange(1, nnz + 1, dtype=np.float64), idx, ptr), shape=(M, M)).T.tocsr()
    at.sort_indices()
    perm = at.data.astype(np.int64) - 1
    want = O.spmm_f32(at.indptr.astype(np.int32), at.indices.astype(np.int32), val[perm], dc, K)
    assert np.array_equal(got.view(np.int32), want.view(np.int32))
    assert np.allclose(ab, O.spmm_abssum(at.indptr.astype(np.int32), at.indices.astype(np.int32), val[perm], dc, K), rtol=1e-12)
