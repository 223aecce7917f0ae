"""Edge softmax without a device: the C restatement of the kernels' order and exp routine (tests/softmax_oracle.c)
against an independent numpy restatement, both against fp64, the exp contract over every float32 in [-87.5, 0], the
status codes of spmm_b200_edge_softmax / _backward and the C++ adapter's new methods."""
import ctypes
import os

import numpy as np
import pytest

from conftest import ROOT
import softmax_oracle as SM

F32, F64 = np.float32, np.float64
TILE = 256


def _ftz(x):
    x = np.asarray(x, F32)
    return np.where(np.abs(x) < np.finfo(F32).tiny, np.copysign(F32(0), x), x).astype(F32)


def _fma32(a, b, c):
    """Correctly rounded float32 fma: the product is exact in fp64, the sum is exact as hi + lo (two-sum); rounding hi
    to float32 can only go wrong when hi is a float32 midpoint, where lo decides."""
    a, b, c = (np.asarray(v, F32) for v in (a, b, c))
    p = a.astype(F64) * b.astype(F64)
    c64 = c.astype(F64)
    hi = p + c64
    bb = hi - p
    lo = (p - (hi - bb)) + (c64 - bb)
    with np.errstate(over="ignore", invalid="ignore"):
        r = hi.astype(F32)
        up = np.nextafter(r, F32(np.inf))
        dn = np.nextafter(r, F32(-np.inf))
        mid_up = hi == (r.astype(F64) + up.astype(F64)) / 2
        mid_dn = hi == (r.astype(F64) + dn.astype(F64)) / 2
    r = np.where(mid_up & (lo > 0), up, r)
    r = np.where(mid_dn & (lo < 0), dn, r)
    return r.astype(F32)


class _Arith:
    """float32 arithmetic of the engine's build: with ftz, every operation flushes subnormal inputs and outputs."""

    def __init__(self, ftz):
        self.fl = _ftz if ftz else (lambda v: np.asarray(v, F32))

    def fma(self, a, b, c):
        return self.fl(_fma32(self.fl(a), self.fl(b), self.fl(c)))

    def add(self, a, b):
        return self.fl(self.fl(a) + self.fl(b))

    def sub(self, a, b):
        return self.fl(self.fl(a) - self.fl(b))

    def mul(self, a, b):
        return self.fl(self.fl(a) * self.fl(b))

    def div(self, a, b):
        return self.fl(self.fl(a) / self.fl(b))


def exp_numpy(x, ftz):
    """The exp routine of edge_softmax.cu, vectorised."""
    A = _Arith(ftz)
    x = np.asarray(x, F32)
    ok = x >= F32(-88.0)
    xx = np.where(ok, x, F32(0))
    kf = A.sub(A.fma(xx, F32(1.44269504), F32(12582912.0)), F32(12582912.0))
    k = kf.astype(np.int32)
    ok &= k >= -126
    r = A.fma(kf, F32(-0.693145751953125), xx)
    r = A.fma(kf, F32(-1.428606765330187e-6), r)
    p = np.full_like(r, F32(1.98412698e-4))
    for coef in (1.38888889e-3, 8.33333333e-3, 4.16666667e-2, 1.66666667e-1, 0.5, 1.0, 1.0):
        p = A.fma(p, r, F32(coef))
    scale = (np.where(ok, k + 127, 127).astype(np.uint32) << 23).view(F32)
    y = A.mul(p, scale)
    y = np.where(y < np.finfo(F32).tiny, F32(0), y)
    return np.where(ok, y, F32(0)).astype(F32)


def _row_sum(terms_a, terms_b, A, bwd):
    """Tiles of 256, lane chains over l + 32 j, xor butterfly, tile sums added from 0.0f in tile order."""
    n = len(terms_a)
    total = F32(0)
    for t0 in range(0, n, TILE):
        c = np.zeros(32, F32)
        for j in range(TILE // 32):
            pos = t0 + j * 32 + np.arange(32)
            ok = pos < n
            pc = np.where(ok, pos, 0)
            new = A.fma(terms_a[pc], terms_b[pc], c) if bwd else A.add(c, terms_a[pc])
            c = np.where(ok, new, c)
        for o in (16, 8, 4, 2, 1):
            c = A.add(c, c[np.arange(32) ^ o])
        total = A.add(total, c[0])
    return F32(total)


def softmax_numpy(ptr, s, ftz):
    A = _Arith(ftz)
    out = np.empty(int(ptr[-1]), F32)
    for r in range(len(ptr) - 1):
        x = s[ptr[r]:ptr[r + 1]]
        if len(x) == 0:
            continue
        if np.any(np.isnan(x) | (x == np.inf)):
            out[ptr[r]:ptr[r + 1]] = np.array(0x7FFFFFFF, np.uint32).view(F32)
            continue
        m = x.max()
        if m == -np.inf:
            out[ptr[r]:ptr[r + 1]] = 0
            continue
        e = exp_numpy(A.sub(x, m), ftz)
        out[ptr[r]:ptr[r + 1]] = A.div(e, _row_sum(e, None, A, False))
    return out


def softmax_backward_numpy(ptr, p, dp, ftz):
    A = _Arith(ftz)
    ds = np.empty(int(ptr[-1]), F32)
    for r in range(len(ptr) - 1):
        a, b = p[ptr[r]:ptr[r + 1]], dp[ptr[r]:ptr[r + 1]]
        if len(a):
            ds[ptr[r]:ptr[r + 1]] = A.mul(a, A.sub(b, _row_sum(a, b, A, True)))
    return ds


def same_bits(a, b):
    """Bit-equal, except that any two NaNs match (the NaN a row holds is documented; NaNs that arithmetic propagates
    keep a payload the CPU and the GPU may choose differently)."""
    a, b = np.asarray(a, F32), np.asarray(b, F32)
    both_nan = np.isnan(a) & np.isnan(b)
    return a.shape == b.shape and bool(np.all(both_nan | (a.view(np.int32) == b.view(np.int32))))


def _case(seed):
    """A random CSR (empty rows, rows that cross tiles and the 1024-entry warp limit) with special rows appended."""
    rng = np.random.default_rng(seed)
    deg = rng.integers(0, 40, 60)
    deg[rng.random(60) < 0.25] = 0
    deg[[3, 17, 29]] = [257, 1025, 2900]
    special = {"ninf": 9, "all_ninf": 5, "nan": 12, "pinf": 7, "subnormal": 300, "single": 1, "big": 40}
    deg = np.concatenate([deg, list(special.values())])
    ptr = np.concatenate([[0], np.cumsum(deg)]).astype(np.int32)
    s = (rng.standard_normal(int(ptr[-1])) * 3).astype(F32)
    rows = {name: 60 + i for i, name in enumerate(special)}
    sl = lambda name: slice(ptr[rows[name]], ptr[rows[name] + 1])
    s[sl("ninf")][::2] = -np.inf
    s[sl("all_ninf")] = -np.inf
    s[sl("nan")][4] = np.nan
    s[sl("pinf")][2] = np.inf
    sub = s[sl("subnormal")]
    sub[:] = (rng.standard_normal(len(sub)) * 1e-39).astype(F32)
    sub[::7] = F32(-1e-30)
    s[sl("big")] = (rng.standard_normal(40) * 40).astype(F32)   # exps that flush below FLT_MIN
    s[ptr[3]:ptr[4]][100] = -np.inf
    return ptr, s, rows


@pytest.mark.parametrize("ftz", [False, True])
@pytest.mark.parametrize("seed", [0, 1])
def test_forward_c_equals_numpy_and_fp64(ftz, seed):
    ptr, s, rows = _case(seed)
    got = SM.edge_softmax_f32(ptr, s, ftz=ftz, nthreads=2)
    assert same_bits(got, softmax_numpy(ptr, s, ftz))
    for r in range(len(ptr) - 1):
        x, o = s[ptr[r]:ptr[r + 1]].astype(F64), got[ptr[r]:ptr[r + 1]]
        if len(x) == 0:
            continue
        if r == rows["nan"] or r == rows["pinf"]:
            assert np.all(o.view(np.uint32) == 0x7FFFFFFF)
        elif r == rows["all_ninf"]:
            assert np.all(o.view(np.uint32) == 0)
        else:
            e = np.exp(x - x.max())
            ref = e / e.sum()
            assert np.all(np.abs(o - ref) <= 4e-6 * ref + 1e-37), r
            assert np.all(o[x == -np.inf].view(np.uint32) == 0)
    assert got[ptr[rows["single"]]] == 1.0


@pytest.mark.parametrize("ftz", [False, True])
@pytest.mark.parametrize("seed", [0, 1])
def test_backward_c_equals_numpy_and_fp64(ftz, seed):
    ptr, s, rows = _case(seed)
    rng = np.random.default_rng(100 + seed)
    p = SM.edge_softmax_f32(ptr, s, ftz=ftz)
    dp = rng.standard_normal(len(p)).astype(F32)
    dp[ptr[rows["subnormal"]]:ptr[rows["subnormal"] + 1]] *= F32(1e-36)   # products that flush
    got = SM.edge_softmax_backward_f32(ptr, p, dp, ftz=ftz, nthreads=2)
    assert same_bits(got, softmax_backward_numpy(ptr, p, dp, ftz))
    for r in range(len(ptr) - 1):
        if r in (rows["nan"], rows["pinf"]) or ptr[r] == ptr[r + 1]:
            continue
        a, b = p[ptr[r]:ptr[r + 1]].astype(F64), dp[ptr[r]:ptr[r + 1]].astype(F64)
        d = (a * b).sum()
        ref = a * (b - d)
        bound = 1e-5 * np.abs(a) * (np.abs(b) + np.abs(a * b).sum()) + 1e-37
        assert np.all(np.abs(got[ptr[r]:ptr[r + 1]] - ref) <= bound), r
    assert np.all(np.isnan(got[ptr[rows["nan"]]:ptr[rows["nan"] + 1]]))   # a NaN row of p stays NaN


@pytest.mark.parametrize("ftz", [False, True])
def test_exp_c_equals_numpy(ftz):
    rng = np.random.default_rng(3)
    x = np.concatenate([-np.abs(rng.standard_normal(200000) * 30), -rng.random(20000) * 1e-37,
                        [0.0, -0.0, -np.inf, -87.3365, -87.33654, -87.5, -88.0, -88.1, -100, -1e-45, -2e-39]]).astype(F32)
    got = SM.softmax_exp(x, ftz)
    assert same_bits(got, exp_numpy(x, ftz))
    assert got[-11] == 1.0 and got[-10] == 1.0 and got[-9] == 0.0


@pytest.mark.parametrize("ftz", [True, False])
def test_exp_contract_exhaustive(ftz):
    """Every float32 in [-87.5, 0]: within 2 ulp of fp64 exp, exp(+-0) == 1, never subnormal, +0 below FLT_MIN."""
    checked, bad, worst = SM.softmax_exp_check(ftz)
    assert checked == 0xC2AF0000 - 0x80000000 + 2
    assert bad == 0
    assert worst <= 2.0


def test_fma_model_rounds_once():
    a = np.array([1 + 2 ** -12], F32)
    c = np.array([-(1 + 2 ** -11)], F32)
    assert _fma32(a, a, c)[0] == F32(2 ** -24)
    assert (a * a + c)[0] == F32(0)


# ---- the C ABI without a device ----------------------------------------------------------------------------------

def test_status_codes_without_gpu():
    from hpc_b200._lib import lib
    assert lib.spmm_b200_edge_softmax(None, None, None, None) == -1
    assert b"null handle" in lib.spmm_b200_last_error()
    assert lib.spmm_b200_edge_softmax_backward(None, None, None, None, None) == -1
    assert b"null handle" in lib.spmm_b200_last_error()
    h = ctypes.c_void_p()
    dummy = (ctypes.c_int * 6)()
    assert lib.spmm_b200_create(dummy, None, None, 5, 0, 32, ctypes.byref(h)) == 0   # num_e = 0: no CUDA call
    assert lib.spmm_b200_edge_softmax(h, None, None, None) == 0
    assert lib.spmm_b200_edge_softmax_backward(h, None, None, None, None) == 0
    assert lib.spmm_b200_destroy(h) == 0
    ptr = (ctypes.c_int * 3)(0, 1, 2)
    idx = (ctypes.c_int * 2)(0, 1)
    val = (ctypes.c_float * 2)(1, 2)
    buf = (ctypes.c_float * 2)()
    assert lib.spmm_b200_create(ptr, idx, val, 2, 2, 32, ctypes.byref(h)) == 0        # no preprocess needed to check
    assert lib.spmm_b200_edge_softmax(h, None, buf, None) == -1
    assert b"null" in lib.spmm_b200_last_error()
    assert lib.spmm_b200_edge_softmax(h, buf, None, None) == -1
    assert lib.spmm_b200_edge_softmax_backward(h, buf, buf, None, None) == -1
    assert lib.spmm_b200_edge_softmax_backward(h, None, buf, buf, None) == -1
    assert lib.spmm_b200_edge_softmax_backward(h, buf, None, buf, None) == -1
    assert b"null" in lib.spmm_b200_last_error()
    assert lib.spmm_b200_destroy(h) == 0


def test_cpp_adapter_edge_softmax_compiles(tmp_path):
    import shutil
    import subprocess
    if not shutil.which("nvcc"):
        pytest.skip("nvcc not on PATH")
    tu = tmp_path / "t.cu"
    tu.write_text('#include "spmm_b200.hpp"\n'
                  'void att(SpMMB200 *a, const float *s, float *p, const float *dp, float *ds) {\n'
                  '    a->edge_softmax(s, p);\n    a->edge_softmax_backward(p, dp, ds);\n}\n')
    r = subprocess.run(["nvcc", "-std=c++14", "-w", "-c", "-o", str(tmp_path / "t.o"), "-I", os.path.join(ROOT, "include"),
                        "-I", os.path.join(ROOT, "hpc_b200", "cpp"), str(tu)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
