"""amax / amin reduce without a device: the C restatement (tests/reduce_oracle.c) against torch.sparse.mm's CPU kernels
and their autograd, the tie / NaN / empty-row rules on hand-built rows, the backward's tile order against a numpy
restatement, the status codes of spmm_b200_reduce / spmm_b200_reduce_backward, the header and the C++ adapter, and the
dispatch coverage of the GPU tests' widths."""
import ctypes
import os
import re
import subprocess

import numpy as np
import pytest

from conftest import ROOT, tiny_csr
import reduce_oracle as RO

torch = pytest.importorskip("torch")

F32, F64 = np.float32, np.float64


def _tie_free_csr(rng, m, b_rows, max_deg):
    """Unique columns per row, some empty rows, edge values normal with a few exact zeros and negatives (at most one
    zero per row, so that no two messages of a row can tie)."""
    ptr, idx = [0], []
    for _ in range(m):
        d = 0 if rng.random() < 0.2 else int(rng.integers(1, max_deg + 1))
        idx.extend(sorted(rng.choice(b_rows, size=min(d, b_rows), replace=False).tolist()))
        ptr.append(len(idx))
    ptr, idx = np.asarray(ptr, np.int32), np.asarray(idx, np.int32)
    val = rng.standard_normal(len(idx)).astype(F32)
    for r in range(m):
        if ptr[r + 1] > ptr[r] and rng.random() < 0.3:
            val[ptr[r]] = 0.0
    return ptr, idx, val


@pytest.mark.parametrize("op", ["amax", "amin"])
@pytest.mark.parametrize("k", [1, 3, 8])
def test_oracle_matches_torch_sparse_mm_and_its_gradients(op, k):
    rng = np.random.default_rng(40 + k)
    m, b_rows = 17, 13
    ptr, idx, val = _tie_free_csr(rng, m, b_rows, 6)
    b = rng.standard_normal((b_rows, k)).astype(F32)
    w = rng.standard_normal((m, k)).astype(F32)
    vout, arg = RO.reduce_f32(ptr, idx, val, b, k, op, ftz=False)
    tv = torch.from_numpy(val.copy()).requires_grad_(True)
    tb = torch.from_numpy(b.copy()).requires_grad_(True)
    a = torch.sparse_csr_tensor(torch.from_numpy(ptr).long(), torch.from_numpy(idx).long(), tv, size=(m, b_rows))
    c = torch.sparse.mm(a, tb, op)
    (c * torch.from_numpy(w)).sum().backward()
    assert np.array_equal(vout, c.detach().numpy())
    deg = np.diff(ptr)
    assert np.all(arg[deg == 0] == -1) and np.all(vout[deg == 0] == 0)
    db, dval = RO.reduce_backward_f32(ptr, idx, val, w, arg, b, b_rows, k, ftz=False)
    assert np.allclose(db, tb.grad.numpy(), rtol=1e-6, atol=1e-7)
    assert np.allclose(dval, tv.grad.numpy(), rtol=1e-6, atol=1e-7)
    f64 = RO.reduce_backward_f64(ptr, idx, val, w, arg, b, b_rows, k)
    assert np.all(np.abs(db - f64["db"]) <= 1e-6 * f64["db_abs"])
    assert np.all(np.abs(dval - f64["dval"]) <= 1e-6 * f64["dval_abs"])


NAN, INF = float("nan"), float("inf")


def _reduce(rows, vin, op, b_rows=None):
    ptr, idx, val = tiny_csr(rows)
    vin = np.asarray(vin, F32).reshape(-1, 1)
    return RO.reduce_f32(ptr, idx, val, vin, 1, op)


@pytest.mark.parametrize("op", ["amax", "amin"])
def test_ties_go_to_the_smaller_position(op):
    vin = [2.0, 3.0, 0.0, -0.0, 1.5]
    # row 0: duplicate column 1 twice with the same value; row 1: 2*3 == 3*2 at positions 2 and 3 (amax) or
    # -(..) for amin; row 2: -0 (position 4) vs +0 (position 5); row 3: 0 * x = +0 vs -0 * x = -0
    rows = [[(1, 1.0), (1, 1.0)], [(1, 2.0 if op == "amax" else -2.0), (0, 3.0 if op == "amax" else -3.0)],
            [(3, 1.0), (2, 1.0)], [(0, 0.0), (0, -0.0)]]
    v, a = _reduce(rows, vin, op)
    assert a[:, 0].tolist() == [0, 2, 4, 6]
    assert v[0, 0] == 3.0 and abs(v[1, 0]) == 6.0
    assert np.signbit(v[2, 0]) and not np.signbit(v[3, 0])   # the winner's own bits: -0 at 4, +0 at 6


@pytest.mark.parametrize("op", ["amax", "amin"])
def test_nan_and_infinities(op):
    vin = [1.0, NAN, INF, -INF]
    rows = [[(0, 5.0), (1, 1.0), (0, 7.0), (1, 2.0)],   # the first NaN wins over numbers and a later NaN
            [(2, 1.0), (3, 1.0), (0, 1.0)],               # +inf (amax), -inf (amin)
            [(2, -1.0), (0, 0.5)],                        # -inf message and a number
            [(2, 0.0)]]                                   # 0 * inf = NaN
    v, a = _reduce(rows, vin, op)
    assert np.isnan(v[0, 0]) and a[0, 0] == 1
    assert v[1, 0] == (INF if op == "amax" else -INF) and a[1, 0] == (4 if op == "amax" else 5)
    assert v[2, 0] == (0.5 if op == "amax" else -INF) and a[2, 0] == (8 if op == "amax" else 7)
    assert np.isnan(v[3, 0]) and a[3, 0] == 9


def test_empty_rows_and_flush_to_zero():
    rows = [[], [(0, 1e-20)], []]
    v, a = _reduce(rows, [1e-20], "amax")
    assert a[:, 0].tolist() == [-1, 0, -1] and not np.signbit(v[0, 0]) and not np.signbit(v[2, 0])
    assert v[1, 0] == 0.0                                 # 1e-40 is subnormal: flushed
    v, _ = RO.reduce_f32(*tiny_csr([[(0, 1e-20)]]), np.asarray([[1e-20]], F32), 1, "amax", ftz=False)
    assert v[0, 0] == F32(1e-20) * F32(1e-20) != 0


def _db_numpy(ptr, idx, val, dc, arg, b_rows, k, tile):
    """The db order written out with numpy: per column of A, matching entries in ascending position, fmaf chains in
    tiles, tile sums added in order (fp32 fma through fp64 is exact here: products of the small integers below)."""
    rows = np.repeat(np.arange(len(ptr) - 1), np.diff(ptr))
    db = np.zeros((b_rows, k), F32)
    for c in range(b_rows):
        ks = np.flatnonzero(idx == c)
        total = np.zeros(k, F32)
        for t0 in range(0, len(ks), tile):
            s = np.zeros(k, F32)
            for e in ks[t0:t0 + tile]:
                r = rows[e]
                hit = arg[r] == e
                s = np.where(hit, (s.astype(F64) + F64(val[e]) * dc[r].astype(F64)).astype(F32), s)
            total = (total + s).astype(F32)
        db[c] = total
    return db


def test_backward_tile_order_on_a_long_column():
    """A column of A longer than several tiles: the fp32 result depends on where the tiles cut, and the restatement
    cuts where the numpy one does. Values are chosen so that each tile sum is exact and the order shows in the
    rounding of the tile sums (2^24 + 1 is not a float32)."""
    n = 3 * RO.TILE + 100
    ptr = np.arange(n + 1, dtype=np.int32)            # n rows of one nonzero each, all in column 0
    idx = np.zeros(n, np.int32)
    val = np.ones(n, F32)
    dc = np.ones((n, 2), F32)
    dc[: RO.TILE, 0] = 2.0 ** 14                      # tile 0 sums to 2^24, then + 1s of the later tiles
    arg = np.tile(np.arange(n, dtype=np.int32)[:, None], (1, 2))
    arg[::7, 1] = -1                                  # some entries do not match column 1
    db, _ = RO.reduce_backward_f32(ptr, idx, val, dc, arg, None, 1, 2, dval=False)
    assert np.array_equal(db, _db_numpy(ptr, idx, val, dc, arg, 1, 2, RO.TILE))
    want0 = F32(F32(F32(2.0 ** 24) + F32(RO.TILE)) + F32(RO.TILE)) + F32(100)
    assert db[0, 0] == want0                          # one chain would have lost every + 1 after 2^24


def test_dval_skips_non_matching_terms_in_sddmm_order():
    import sddmm_oracle as SO
    rng = np.random.default_rng(3)
    for k in (3, 8, 36, 132, 516):
        ptr, idx, val = _tie_free_csr(rng, 9, 7, 5)
        b = rng.standard_normal((7, k)).astype(F32)
        dc = rng.standard_normal((9, k)).astype(F32)
        _, arg = RO.reduce_f32(ptr, idx, val, b, k, "amax")
        _, dval = RO.reduce_backward_f32(ptr, idx, val, dc, arg, b, 7, k, db=False)
        rows = np.repeat(np.arange(9), np.diff(ptr))
        for e in range(len(idx)):                     # masking dc by the match gives the same chain (fma with 0 adds 0)
            x = np.where(arg[rows[e]] == e, dc[rows[e]], F32(0))
            want = SO.sddmm_f32(np.array([0, 1], np.int32), idx[e:e + 1], x, b, k)
            assert dval[e].view(np.int32) == want[0].view(np.int32) or (dval[e] == 0 and want[0] == 0)


# ---- the C ABI without a device ----------------------------------------------------------------------------------

def test_status_codes_without_gpu():
    from hpc_b200._lib import lib
    assert lib.spmm_b200_reduce(None, 1, None, None, None, None) == -1
    assert b"null handle" in lib.spmm_b200_last_error()
    assert lib.spmm_b200_reduce_backward(None, None, None, None, None, None, None) == -1
    h = ctypes.c_void_p()
    dummy = (ctypes.c_int * 6)()
    assert lib.spmm_b200_create(dummy, None, None, 5, 0, 32, ctypes.byref(h)) == 0
    assert lib.spmm_b200_reduce(h, 3, None, None, None, None) == -1                # bad op
    assert b"op" in lib.spmm_b200_last_error()
    assert lib.spmm_b200_reduce(h, 0, None, None, None, None) == -1
    assert lib.spmm_b200_reduce(h, 1, None, None, None, None) == -2                # before preprocess
    assert b"preprocess" in lib.spmm_b200_last_error()
    assert lib.spmm_b200_reduce_backward(h, None, None, None, None, None, None) == -1   # not a transposed operator
    assert b"transposed" in lib.spmm_b200_last_error()
    assert lib.spmm_b200_destroy(h) == 0


def test_degenerate_handles_without_gpu():
    """feat_in = 0 and num_v = 0 plans build without a CUDA call; reduce on them returns 0, and set_feat / b_rows
    invalidate it as they invalidate run."""
    from hpc_b200._lib import lib
    h = ctypes.c_void_p()
    dummy = (ctypes.c_int * 6)()
    assert lib.spmm_b200_create(dummy, None, None, 5, 0, 0, ctypes.byref(h)) == 0
    assert lib.spmm_b200_preprocess(h, None, None, None) == 0
    assert lib.spmm_b200_reduce(h, 2, None, None, None, None) == 0
    assert lib.spmm_b200_set_option(h, b"b_rows", 7) == 0
    assert lib.spmm_b200_reduce(h, 2, None, None, None, None) == -2
    assert lib.spmm_b200_preprocess(h, None, None, None) == 0
    assert lib.spmm_b200_set_feat(h, 0) == 0
    assert lib.spmm_b200_reduce(h, 1, None, None, None, None) == -2
    assert lib.spmm_b200_destroy(h) == 0
    assert lib.spmm_b200_create(None, None, None, 0, 0, 32, ctypes.byref(h)) == 0
    assert lib.spmm_b200_preprocess(h, None, None, None) == 0
    assert lib.spmm_b200_reduce(h, 1, None, None, None, None) == 0
    assert lib.spmm_b200_destroy(h) == 0


def test_header_declares_the_entries_in_plain_c(tmp_path):
    tu = tmp_path / "t.c"
    tu.write_text('#include "spmm_b200.h"\n'
                  'int main(void) {\n'
                  '    int (*f)(spmm_b200_t, int, const float *, float *, int *, void *) = spmm_b200_reduce;\n'
                  '    int (*g)(spmm_b200_t, const float *, const int *, const float *, float *, float *, void *) =\n'
                  '        spmm_b200_reduce_backward;\n'
                  '    (void)f; (void)g;\n'
                  '    return SPMM_B200_REDUCE_AMAX + SPMM_B200_REDUCE_AMIN == 3 ? 0 : 1;\n'
                  '}\n')
    r = subprocess.run(["gcc", "-std=c99", "-pedantic", "-Wall", "-Werror", "-fsyntax-only", "-I",
                        os.path.join(ROOT, "include"), str(tu)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr


def test_cpp_adapter_reduce_compiles(tmp_path):
    import shutil
    if not shutil.which("nvcc"):
        pytest.skip("nvcc not on PATH")
    tu = tmp_path / "t.cu"
    tu.write_text('#include "spmm_b200.hpp"\n'
                  'void step(SpMMB200 *a, SpMMB200 *t, const float *b, float *c, int *arg, const float *dc, float *db,\n'
                  '          float *dval) {\n'
                  '    a->reduce(SPMM_B200_REDUCE_AMAX, b, c, arg);\n'
                  '    t->reduce_backward(dc, arg, b, db, dval);\n'
                  '}\n')
    r = subprocess.run(["nvcc", "-std=c++14", "-w", "-c", "-o", str(tmp_path / "t.o"), "-I", os.path.join(ROOT, "include"),
                        "-I", os.path.join(ROOT, "hpc_b200", "cpp"), str(tu)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr


# ---- dispatch coverage of the GPU tests ----------------------------------------------------------------------------

def _layout(k):
    """layout() of reduce.cu: (W columns per unit, lanes, units per lane and slice, slices)"""
    def pow2(q):
        lanes = 1
        while lanes < q and lanes < 32:
            lanes <<= 1
        return lanes
    if k % 4 == 0 and k <= 512:
        q = k // 4
        lanes = pow2(q)
        need = -(-q // lanes)
        w, vec = 4, 1 if need <= 1 else 2 if need <= 2 else 4
    elif k % 4 == 0:
        w, lanes, vec = 4, 32, 4
    else:
        w, lanes, vec = 1, pow2(k), 4
    return w, lanes, vec, -(-k // (lanes * vec * w))


def test_gpu_widths_reach_every_reduce_dispatch_case():
    """The widths of tests/test_reduce_gpu.py launch every (W, VEC) instantiation of reduce.cu's dispatch (read from
    the source), float4 shapes at every lane count, one-slice and several-slice float4 and scalar layouts, and scalar
    layouts at every lane count."""
    import test_reduce_gpu as RG
    src = open(os.path.join(ROOT, "hpc_b200", "csrc", "reduce.cu")).read()
    table = {(int(w), int(v)) for w, v in re.findall(r"launch_fwd<(\d+), (\d+), \d+>\(a, gr, s\)", src)}
    assert table == {(4, 1), (4, 2), (4, 4), (1, 4)}
    assert table == {(int(w), int(v)) for w, v in re.findall(r"launch_bwd<(\d+), (\d+), \d+>\(a, gr, s\)", src)}
    shapes = [_layout(k) for k in RG.WIDTHS]
    assert {(w, v) for w, _, v, _ in shapes} == table
    assert {lanes for w, lanes, v, _ in shapes if w == 4 and v == 1} == {1, 2, 4, 8, 16, 32}
    assert {lanes for w, lanes, _, _ in shapes if w == 1} == {1, 2, 4, 8, 16, 32}
    assert {(w, n > 1) for w, _, _, n in shapes} == {(4, False), (4, True), (1, False), (1, True)}
    assert 1024 in RG.WIDTHS and 516 in RG.WIDTHS


def test_path_tests_reach_every_reduce_boundary():
    """tests/test_reduce_paths_gpu.py reaches, with the thresholds read from reduce.cu and rows.cuh: every (W, VEC)
    instantiation of the forward (its CTA kernel included) at every float4 lane count, one- and several-slice layouts;
    rows on each side of kWarpMax; Aᵀ rows on each side of kTile and kBwdWarpMax; and a second round of the backward
    CTA's lane groups at L = 1, 4, 8 and 32, ending partway through it."""
    import test_reduce_paths_gpu as RP
    src = open(os.path.join(ROOT, "hpc_b200", "csrc", "reduce.cu")).read()
    rows_src = open(os.path.join(ROOT, "hpc_b200", "csrc", "rows.cuh")).read()
    c = RP.source_constants()
    assert f"constexpr int kWarpMax = {c['kWarpMax']};" in src and f"constexpr int kTile = {c['kTile']};" in src
    assert "constexpr int kBwdWarpMax = 4 * kTile;" in src and c["kBwdWarpMax"] == 4 * c["kTile"]
    assert f"constexpr int kRowBlock = {c['kRowBlock']};" in rows_src and c["kRowWarps"] == c["kRowBlock"] // 32
    table = {(int(w), int(v)) for w, v in re.findall(r"launch_fwd<(\d+), (\d+), \d+>\(a, gr, s\)", src)}
    fwd = [_layout(k) for k in RP.FWD_WIDTHS]
    assert {(w, v) for w, _, v, _ in fwd} == table
    assert {lanes for w, lanes, _, _ in fwd if w == 4} == {1, 2, 4, 8, 16, 32}
    assert {lanes for w, lanes, _, _ in fwd if w == 1} >= {1, 32}
    assert {(w, n > 1) for w, _, _, n in fwd} == {(4, False), (4, True), (1, False), (1, True)}
    lens = set(RP.FWD_ROW_LENGTHS)
    assert {c["kWarpMax"] - 1, c["kWarpMax"], c["kWarpMax"] + 1} <= lens and max(lens) >= 30 * c["kWarpMax"]
    cols = RP.BWD_COLUMN_LENGTHS
    T, W = c["kTile"], c["kBwdWarpMax"]
    assert {T - 1, T, T + 1, W, W + 1} <= set(cols)
    bwd_lanes = {_layout(k)[1] for k in RP.BWD_WIDTHS}
    assert bwd_lanes >= {1, 4, 8, 32}
    assert any(_layout(k)[3] > 1 for k in RP.BWD_WIDTHS)                 # the separate dval walk
    for lanes in (1, 4, 8, 32):
        workers = c["kRowWarps"] * 32 // lanes
        tiles = [-(-n // T) for n in cols]
        assert any(t > workers and t % workers for t in tiles), lanes     # a second round, the last one partial
    assert c["kRowWarps"] * 32 // 32 * T in cols                          # exactly one full round at L = 32
