"""SDDMM without a device: the C restatement of the kernel's order (tests/sddmm_oracle.c) against an independent numpy
restatement, both against fp64, the status codes of spmm_b200_sddmm and the C++ adapter's new method."""
import ctypes
import os

import numpy as np
import pytest

from conftest import ROOT
import sddmm_oracle as SO

F32, F64 = np.float32, np.float64


def _ftz(x):
    x = np.asarray(x, F32)
    return np.where(np.abs(x) < np.finfo(F32).tiny, np.copysign(F32(0), x), x).astype(F32)


def _fma32(a, b, c):
    """Correctly rounded float32 fma: the product is exact in fp64, the sum is exact as hi + lo (two-sum); rounding hi
    to float32 can only go wrong when hi is a float32 midpoint, where lo decides."""
    p = a.astype(F64) * b.astype(F64)
    c64 = c.astype(F64)
    hi = p + c64
    bb = hi - p
    lo = (p - (hi - bb)) + (c64 - bb)
    with np.errstate(over="ignore"):
        r = hi.astype(F32)
        up = np.nextafter(r, F32(np.inf))
        dn = np.nextafter(r, F32(-np.inf))
    mid_up = hi == (r.astype(F64) + up.astype(F64)) / 2
    mid_dn = hi == (r.astype(F64) + dn.astype(F64)) / 2
    r = np.where(mid_up & (lo > 0), up, r)
    r = np.where(mid_dn & (lo < 0), dn, r)
    return r.astype(F32)


def sddmm_numpy(ptr, idx, x_row, x_col, k, ftz):
    """The order of hpc_b200/csrc/sddmm.cu, vectorised over the nonzeros and the lanes."""
    nnz = int(ptr[-1])
    rows = np.repeat(np.arange(len(ptr) - 1), np.diff(ptr))
    xr = x_row.reshape(-1, k)[rows] if k else np.zeros((nnz, 0), F32)
    xc = x_col.reshape(-1, k)[idx] if k else np.zeros((nnz, 0), F32)
    w = 4 if k % 4 == 0 else 1
    q_n = k // w
    lanes = 1
    while lanes < q_n and lanes < 32:
        lanes *= 2
    fl = _ftz if ftz else (lambda v: v)
    s = np.zeros((nnz, lanes), F32)
    for step in range((q_n + lanes - 1) // lanes):
        q = np.arange(lanes) + step * lanes
        ok = q < q_n
        for t in range(w):
            col = np.where(ok, q * w + t, 0)
            new = fl(_fma32(fl(xr[:, col]), fl(xc[:, col]), fl(s)))
            s = np.where(ok[None, :], new, s)
    o = lanes // 2
    while o:
        s = fl(fl(s) + fl(s[:, np.arange(lanes) ^ o])).astype(F32)
        o //= 2
    return s[:, 0].copy()


def _random_csr(rng, m, b_rows, max_deg):
    deg = rng.integers(0, max_deg + 1, m)
    deg[rng.random(m) < 0.25] = 0                       # empty rows
    ptr = np.concatenate([[0], np.cumsum(deg)]).astype(np.int32)
    idx = rng.integers(0, b_rows, int(ptr[-1])).astype(np.int32)   # unsorted, with duplicates
    if len(idx) > 2:
        idx[1] = idx[0]
    return ptr, idx


KS = [0, 1, 3, 4, 8, 12, 32, 36, 96, 128, 256, 260, 512]


@pytest.mark.parametrize("k", KS)
@pytest.mark.parametrize("ftz", [False, True])
def test_c_restatement_equals_numpy_and_fp64(k, ftz):
    rng = np.random.default_rng(1000 + k)
    m, b_rows = 23, 31
    ptr, idx = _random_csr(rng, m, b_rows, 9)
    x_row = rng.standard_normal(m * k).astype(F32)
    x_col = rng.standard_normal(b_rows * k).astype(F32)
    if k:   # subnormal inputs, and products that underflow
        x_row[rng.random(m * k) < 0.1] = F32(3e-39)
        x_col[rng.random(b_rows * k) < 0.1] = F32(-2e-39)
        x_col[rng.random(b_rows * k) < 0.05] = F32(1e-30)
    got = SO.sddmm_f32(ptr, idx, x_row, x_col, k, ftz=ftz, nthreads=2)
    ref = sddmm_numpy(ptr, idx, x_row, x_col, k, ftz)
    assert got.shape == (int(ptr[-1]),)
    assert np.array_equal(got.view(np.int32), ref.view(np.int32))
    d64, ab = SO.sddmm_f64(ptr, idx, x_row, x_col, k)
    assert np.all(np.abs(got.astype(F64) - d64) <= 1e-5 * ab + 1e-30)
    if k == 0:
        assert np.all(got.view(np.int32) == 0)            # +0.0f


def test_fma_model_rounds_once():
    """The numpy fma is correctly rounded where a multiply-then-add would round twice."""
    a = np.array([1 + 2 ** -12], F32)
    c = np.array([-(1 + 2 ** -11)], F32)
    # a*a = 1 + 2^-11 + 2^-24: the product alone rounds to 1 + 2^-11, the fma keeps the 2^-24
    assert _fma32(a, a, c)[0] == F32(2 ** -24)
    assert (a * a + c)[0] == F32(0)


# ---- the C ABI without a device ----------------------------------------------------------------------------------

def test_status_codes_without_gpu():
    from hpc_b200._lib import lib
    assert lib.spmm_b200_sddmm(None, None, None, None, None) == -1
    assert b"null handle" in lib.spmm_b200_last_error()
    h = ctypes.c_void_p()
    dummy = (ctypes.c_int * 6)()
    assert lib.spmm_b200_create(dummy, None, None, 5, 0, 32, ctypes.byref(h)) == 0
    assert lib.spmm_b200_sddmm(h, None, None, None, None) == -2          # before preprocess
    assert b"preprocess" in lib.spmm_b200_last_error()
    assert lib.spmm_b200_destroy(h) == 0


def test_degenerate_handles_without_gpu():
    """feat_in = 0 and num_e = 0 plans build without a CUDA call; sddmm on them is a no-op returning 0, and set_feat /
    b_rows invalidate it as they invalidate run."""
    from hpc_b200._lib import lib
    h = ctypes.c_void_p()
    dummy = (ctypes.c_int * 6)()
    assert lib.spmm_b200_create(dummy, None, None, 5, 0, 0, ctypes.byref(h)) == 0      # feat_in = 0, num_e = 0
    assert lib.spmm_b200_preprocess(h, None, None, None) == 0
    assert lib.spmm_b200_sddmm(h, None, None, None, None) == 0
    assert lib.spmm_b200_set_option(h, b"b_rows", 7) == 0
    assert lib.spmm_b200_sddmm(h, None, None, None, None) == -2
    assert lib.spmm_b200_preprocess(h, None, None, None) == 0
    assert lib.spmm_b200_set_feat(h, 0) == 0
    assert lib.spmm_b200_sddmm(h, None, None, None, None) == -2
    assert lib.spmm_b200_destroy(h) == 0
    assert lib.spmm_b200_create(None, None, None, 0, 0, 32, ctypes.byref(h)) == 0     # no rows, feat_in = 32
    assert lib.spmm_b200_preprocess(h, None, None, None) == 0
    assert lib.spmm_b200_sddmm(h, None, None, None, None) == 0
    assert lib.spmm_b200_destroy(h) == 0


def test_null_output_without_gpu():
    """With nonzeros, a null out (or null inputs at feat_in > 0) is EINVAL before any CUDA call."""
    from hpc_b200._lib import lib
    h = ctypes.c_void_p()
    ptr = (ctypes.c_int * 3)(0, 1, 2)
    idx = (ctypes.c_int * 2)(0, 1)
    val = (ctypes.c_float * 2)(1, 2)
    assert lib.spmm_b200_create(ptr, idx, val, 2, 2, 0, ctypes.byref(h)) == 0
    assert lib.spmm_b200_preprocess(h, None, None, None) == 0                         # feat_in = 0: no CUDA call
    assert lib.spmm_b200_sddmm(h, None, None, None, None) == -1
    assert b"null" in lib.spmm_b200_last_error()
    assert lib.spmm_b200_destroy(h) == 0


def test_cpp_adapter_sddmm_compiles(tmp_path):
    import shutil
    import subprocess
    if not shutil.which("nvcc"):
        pytest.skip("nvcc not on PATH")
    tu = tmp_path / "t.cu"
    tu.write_text('#include "spmm_b200.hpp"\n'
                  'void grad(SpMMB200 *a, const float *dc, const float *b, float *dval) { a->sddmm(dc, b, dval); }\n')
    r = subprocess.run(["nvcc", "-std=c++14", "-w", "-c", "-o", str(tmp_path / "t.o"), "-I", os.path.join(ROOT, "include"),
                        "-I", os.path.join(ROOT, "hpc_b200", "cpp"), str(tu)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr


# ---- dispatch coverage of the GPU tests ----------------------------------------------------------------------------

def _pow2_lanes(q):
    """pow2_lanes of common.h (the lane count of sddmm.cu and reduce.cu)"""
    lanes = 1
    while lanes < q and lanes < 32:
        lanes <<= 1
    return lanes


def _fast_shape(k):
    """fast_lane_shape of common.h: (lanes, float4 per lane) of sddmm_kernel for K % 4 == 0, K <= 512"""
    q = k // 4
    lanes = _pow2_lanes(q)
    need = -(-q // lanes)
    return lanes, 1 if need <= 1 else 2 if need <= 2 else 4


def test_kernel_path_widths_reach_every_sddmm_dispatch_case():
    """The widths of tests/test_kernel_paths_gpu.py launch every sddmm_kernel<LANES, VEC, U> in sddmm.cu's dispatch table
    (read from the source, so a new case without a width fails here), each with all float4 slots of its lanes used and,
    where the lane count leaves room (LANES >= 4), with some unused; sddmm_generic_kernel<true> (K > 512); and
    sddmm_generic_kernel<false> at every lane count 1 .. 32."""
    import re
    import test_kernel_paths_gpu as KP
    src = open(os.path.join(ROOT, "hpc_b200", "csrc", "sddmm.cu")).read()
    table = {(int(l), int(v)) for l, v in re.findall(r"case \d+: return fast_fn<(\d+), (\d+), \d+>\(\);", src)}
    assert len(table) == 8
    full, partial = set(), set()
    for k in KP.SDDMM_FAST_WIDTHS:
        assert k % 4 == 0 and 0 < k <= 512
        lanes, vec = _fast_shape(k)
        (full if k // 4 == lanes * vec else partial).add((lanes, vec))
    assert full == table
    assert partial == {s for s in table if s[0] >= 4}
    assert all(k % 4 == 0 and k > 512 for k in KP.SDDMM_GENERIC_V4_WIDTHS)
    scalar = KP.SDDMM_GENERIC_SCALAR_WIDTHS
    assert all(k % 4 != 0 for k in scalar)
    assert {_pow2_lanes(k) for k in scalar} == {1, 2, 4, 8, 16, 32}
    assert any(_pow2_lanes(k) == 32 and k > 32 for k in scalar)          # a lane walks more than one column
    assert set(KP.SDDMM_WIDTHS) == set(KP.SDDMM_FAST_WIDTHS + KP.SDDMM_GENERIC_V4_WIDTHS + scalar)
