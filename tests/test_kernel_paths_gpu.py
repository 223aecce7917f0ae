"""Every dispatch entry of the SDDMM, edge-softmax and autograd kernels against fp64, at the shapes where kernels go wrong.

Two bars per case: bit-exact against the CPU restatement of the documented order (tests/sddmm_oracle.c,
tests/softmax_oracle.c, oracle/spmm_oracle.c), and within a bound on the distance to the fp64 result that is derived
from that order (not a chosen constant). The widths below are chosen so that every kernel instantiation is launched;
tests/test_sddmm_oracle.py checks that they reach every dispatch case of sddmm.cu.

The cases past 2^31 elements need tens of GB and skip, naming the bytes, where the device or host has less free.
"""
import ctypes as C
import gc
import math
import os

import numpy as np
import pytest

torch = pytest.importorskip("torch")

import hpc_b200 as H  # noqa: E402
from hpc_b200._lib import check, lib  # noqa: E402

HAVE_CUDA = torch.cuda.is_available()
pytestmark = [pytest.mark.gpu, pytest.mark.skipif(not HAVE_CUDA, reason="no CUDA device")]

DEV = "cuda"
F32, F64 = np.float32, np.float64
U = 2.0 ** -24                       # unit roundoff of float32
FLT_MIN = 2.0 ** -126

# SDDMM widths (sddmm.cu): K % 4 == 0 and K <= 512 take sddmm_kernel<L, VEC, U> with Q = K/4, L = min(32, pow2ceil(Q))
# lanes and VEC = ceil(Q/L) float4 per lane rounded up to 1, 2 or 4; every (L, VEC) below is met with all its float4
# slots filled (Q = L*VEC) and, where L > 2 allows it, with some left empty (the qok predicate false).
SDDMM_FAST_WIDTHS = [4, 8, 12, 16, 20, 32, 36, 64, 68, 100, 128, 132, 256, 260, 388, 512]
SDDMM_GENERIC_V4_WIDTHS = [516, 1024]                  # sddmm_generic_kernel<true>, 32 lanes
SDDMM_GENERIC_SCALAR_WIDTHS = [1, 2, 3, 7, 13, 33, 515]  # sddmm_generic_kernel<false>: lanes 1, 2, 4, 8, 16, 32, 32
SDDMM_WIDTHS = SDDMM_FAST_WIDTHS + SDDMM_GENERIC_V4_WIDTHS + SDDMM_GENERIC_SCALAR_WIDTHS

# autograd: scalar SpMM + generic scalar SDDMM (7, 33), sddmm_kernel<32, 1, 4> (128), multi-slice SpMM + generic float4
# SDDMM (516)
AUTOGRAD_WIDTHS = [7, 33, 128, 516]


@pytest.fixture(autouse=True)
def _release_memory():
    yield
    gc.collect()
    if HAVE_CUDA:
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        H.trim_memory()


# ---- helpers -----------------------------------------------------------------------------------------------------

def _bits_equal(a, b):
    a, b = np.asarray(a, F32), np.asarray(b, F32)
    return a.shape == b.shape and np.array_equal(a.view(np.int32), b.view(np.int32))


def _same(a, b):
    """Bit-equal, NaN matching NaN (whatever its payload)."""
    a, b = np.asarray(a, F32), np.asarray(b, F32)
    return a.shape == b.shape and bool(np.all((np.isnan(a) & np.isnan(b)) | (a.view(np.int32) == b.view(np.int32))))


def _csr(ptr, idx, val=None, seed=7):
    nnz = len(idx)
    d_val = (H.fill_normal(torch.empty(max(nnz, 1), device=DEV), seed, 1) if val is None
             else torch.from_numpy(np.ascontiguousarray(val, F32)).to(DEV))
    return H.CSR(len(ptr) - 1, nnz, torch.from_numpy(np.ascontiguousarray(ptr, np.int32)).to(DEV),
                 torch.from_numpy(np.ascontiguousarray(idx, np.int32)).to(DEV), d_val)


def _dense(n, seed, stream):
    return H.fill_normal(torch.empty(max(n, 1), device=DEV), seed, stream)


def _whole_rows(op, m):
    heavy = _heavy_rows(op)
    return np.setdiff1d(np.arange(m), heavy)


def _heavy_rows(op):
    """Rows split into segments in any column block (their sums are re-associated), read without copying the rest of
    the plan."""
    rows = []
    for b in range(op.plan_info(0)["n_col_blocks"]):
        n = op.plan_info(b)["n_heavy"]
        a = np.empty(n, np.int32)
        if n:
            check(lib.spmm_b200_plan_copy(op._h, 1, a.ctypes.data_as(C.c_void_p), a.nbytes))
        rows.append(a)
    return np.unique(np.concatenate(rows)) if rows else np.zeros(0, np.int32)


def _sub_problem(ptr, idx, rows):
    """The CSR of `rows` alone (same nonzero order) with its columns renumbered over the distinct columns it reads.
    -> (ptr, idx, CSR positions of its nonzeros in the full graph, the full graph's column of each new column)."""
    ptr = np.asarray(ptr, np.int64)
    starts, lens = ptr[rows], ptr[np.asarray(rows) + 1] - ptr[rows]
    sptr = np.concatenate([[0], np.cumsum(lens)])
    pos = np.repeat(starts - sptr[:-1], lens) + np.arange(sptr[-1])
    cols, sidx = np.unique(np.asarray(idx)[pos], return_inverse=True)
    return sptr.astype(np.int32), sidx.astype(np.int32), pos, cols


def _need_memory(device_bytes, host_bytes=0):
    free, _ = torch.cuda.mem_get_info()
    if free < device_bytes:
        pytest.skip(f"needs {device_bytes} bytes ({device_bytes / 2**30:.1f} GiB) of free device memory, "
                    f"{free} free")
    if host_bytes:
        avail = os.sysconf("SC_AVPHYS_PAGES") * os.sysconf("SC_PAGE_SIZE")
        if avail < host_bytes:
            pytest.skip(f"needs {host_bytes} bytes ({host_bytes / 2**30:.1f} GiB) of free host memory, {avail} free")


# ---- the SDDMM order and its error bound -------------------------------------------------------------------------

def _sddmm_lanes(q):
    lanes = 1
    while lanes < q and lanes < 32:
        lanes *= 2
    return lanes


def _sddmm_roundings(K):
    """Roundings a product goes through on its way to out[e] in the documented order (sddmm.cu): W = 4 columns per group
    when K % 4 == 0 (else 1), Q = K / W groups, L lanes; a lane's FMA chain has ceil(Q / L) * W links (each one rounding,
    the first adding to 0.0f exactly), then log2 L butterfly adds."""
    W = 4 if K % 4 == 0 else 1
    Q = K // W
    L = _sddmm_lanes(Q)
    return -(-Q // L) * W + int(math.log2(L))


def _sddmm_bound(K, abs_terms):
    """|got - exact| <= gamma_n * sum |x_row * x_col| + n * 2^-126.

    Every product enters one lane's chain and reaches out[e] through at most n roundings (an FMA rounds product + sum
    once; a butterfly add rounds once). A sum of terms each carried through at most n roundings of relative error <= u
    (round to nearest, u = 2^-24) differs from the exact sum by at most gamma_n * sum |terms| with
    gamma_n = n u / (1 - n u) (Higham, Accuracy and Stability, Lemma 3.1 / eq. 3.5). The build flushes subnormal results
    to zero: each of the n operations can lose one result below 2^-126 outright, an absolute n * 2^-126."""
    n = _sddmm_roundings(K)
    gamma = n * U / (1 - n * U)
    return gamma * abs_terms + n * FLT_MIN


def _check_sddmm(ptr, idx, x_row, x_col, K, got):
    import sddmm_oracle as SO
    assert _bits_equal(got, SO.sddmm_f32(ptr, idx, x_row, x_col, K, ftz=True))
    exact, ab = SO.sddmm_f64(ptr, idx, x_row, x_col, K)
    assert np.all(np.abs(got.astype(F64) - exact) <= _sddmm_bound(K, ab))


# ---- a. SDDMM, every dispatch entry -------------------------------------------------------------------------------

def _crafted_graph(shuffled=False, seed=3):
    """num_v x b_rows (b_rows > num_v) CSR that reaches the SDDMM kernels' branches: empty first and last rows and a run
    of empty rows; runs of 1- and 2-nonzero rows (two new rows inside one batch of entries); rows of many 128-nonzero
    chunks (warps start mid-row); duplicate columns; column b_rows - 1; and column 0 and column b_rows - 1 each read by
    hundreds of rows (long rows of the transposed operator). Columns ascend in every row unless `shuffled`."""
    rng = np.random.default_rng(seed)
    num_v, b_rows = 2000, 2600
    deg = rng.integers(0, 12, num_v)
    deg[0] = deg[-1] = 0
    deg[100:140] = 0
    deg[200:400] = rng.integers(1, 3, 200)
    deg[[500, 900, 1500]] = [700, 1500, 3000]
    ptr = np.concatenate([[0], np.cumsum(deg)]).astype(np.int32)
    idx = np.empty(int(ptr[-1]), np.int32)
    for r in range(num_v):
        d = int(deg[r])
        if not d:
            continue
        hi = 300 if d == 1500 else b_rows          # row 900 reads 300 columns 1500 times: duplicates
        cols = np.sort(rng.integers(0, hi, d))
        if r % 3 == 0:
            cols[-1] = b_rows - 1
        if r % 5 == 0:
            cols[0] = 0
        if shuffled:
            rng.shuffle(cols)
        idx[ptr[r]:ptr[r + 1]] = cols
    return ptr, idx, b_rows


CRAFTED = {}


def _crafted(shuffled=False):
    if shuffled not in CRAFTED:
        CRAFTED[shuffled] = _crafted_graph(shuffled)
    return CRAFTED[shuffled]


@pytest.mark.parametrize("variant", ["col_blocks1", "col_blocks3", "unsorted"])
@pytest.mark.parametrize("K", SDDMM_WIDTHS)
def test_sddmm_every_dispatch_entry(K, variant):
    ptr, idx, b_rows = _crafted(shuffled=variant == "unsorted")
    M = len(ptr) - 1
    blocks = 1 if variant == "col_blocks1" else 3
    g = _csr(ptr, idx)
    xr, xc = _dense(M * K, K, 3), _dense(b_rows * K, K, 4)
    op = H.SpMMB200(g, K, b_rows=b_rows, col_blocks=blocks)
    op.preprocess(xc, torch.empty(M * K, device=DEV))
    # three blocks for sorted rows in the vector kernels; the scalar plan and unsorted rows keep one
    assert op.plan_info()["n_col_blocks"] == (3 if blocks == 3 and K % 4 == 0 and variant != "unsorted" else 1)
    out = torch.full((len(idx),), float("nan"), device=DEV)
    op.sddmm(xr, xc, out)
    torch.cuda.synchronize()
    _check_sddmm(ptr, idx, xr[: M * K].cpu().numpy(), xc[: b_rows * K].cpu().numpy(), K, out.cpu().numpy())
    op.close()


# ---- b. edge softmax at the warp / CTA and stripe boundaries ------------------------------------------------------

WARP_LENGTHS = [255, 256, 511, 512, 768, 1023, 1024]        # one warp per row (<= 4 tiles of 256)
CTA_LENGTHS = [1025, 16383, 16384, 16385, 32769]            # one CTA per row; 16,384 = 64 tiles = one tile-sum round


def _softmax_graph(sms, seed=17):
    """Rows of 0..23 nonzeros with the lengths above placed: in the first grid of the long-row kernel (grid = 4 * SMs
    CTAs of 256-row stripes), beyond it (rows >= 4 * SMs * 256, reached by the stripe loop), at num_v - 1, and two long
    rows inside one 32-row group (one ballot) both in the first grid and beyond it."""
    first = 4 * sms * 256
    num_v = max(160_000, first + 12_288)
    rng = np.random.default_rng(seed)
    deg = rng.integers(0, 24, num_v)
    deg[rng.random(num_v) < 0.2] = 0
    for i, n in enumerate(WARP_LENGTHS):
        deg[1000 + 37 * i] = n
        deg[first + 3000 + 41 * i] = n
    for i, n in enumerate(CTA_LENGTHS):
        deg[5000 + 300 * i] = n                  # first grid
        deg[first + 5 + 700 * i] = n             # beyond it
    deg[[64_000, 64_005]] = [16_385, 1025]       # one 32-row group, first grid
    deg[[first + 6400, first + 6401]] = [32_769, 16_384]   # one 32-row group, beyond it
    deg[first] = 2000                            # first row of the first stripe past the grid
    deg[num_v - 1] = 16_385
    return np.concatenate([[0], np.cumsum(deg)]).astype(np.int32)


def _softmax_fp64(ptr, s):
    """-> (p, m per nonzero, S per nonzero, n per nonzero) in fp64 for finite scores."""
    deg = np.diff(ptr).astype(np.int64)
    rows = np.repeat(np.arange(len(deg)), deg)
    s64 = s.astype(F64)
    nz = np.flatnonzero(deg)
    m = np.full(len(deg), -np.inf)
    m[nz] = np.maximum.reduceat(s64, ptr[:-1][nz])
    e = np.exp(s64 - m[rows])
    S = np.bincount(rows, e, len(deg))
    return e / S[rows], m[rows], S[rows], deg[rows]


def _gamma(n):
    return n * U / (1 - n * U)


def _check_softmax_forward(ptr, s, got):
    """|p_got - p| <= rel * p + 2^-125 per nonzero of a row with max m and n nonzeros (edge_softmax.cu's order).

    x = exp(s - m) is computed as sm_exp(fl(s - m)):
      * fl(s - m) = (s - m)(1 + d), |d| <= u, so exp of it is exp(s - m) * exp(+-u |s - m|);
      * sm_exp is within 2 ulp of exp on [-87.5, 0] (checked exhaustively by tests/test_edge_softmax_oracle.py), and an
        ulp of a normal float y is at most 2^-23 y: relative 4u.
      So x_got = x (1 + e_x) with 1 + e_x <= (1 + 4u) exp(u |s - m|) =: 1 + eta. A result below FLT_MIN is 0 (or FLT_MIN):
      absolute < FLT_MIN.
    S is a sum of positive terms, each through at most 8 (lane chain) + 5 (butterfly) + ceil(n / 256) (tile sums from
    0.0f) roundings: |S_got - sum x_got| <= gamma_nS sum x_got. The largest term is exp(0) = 1 exactly, so S >= 1 and the
    flushed terms add at most n FLT_MIN relative: S_got = S (1 + r), |r| <= rho = (1 + eta_max)(1 + gamma_nS) - 1 +
    n 2^-126. out = fl(x_got / S_got) adds one rounding: p_got / p <= (1 + eta)(1 + u) / (1 - rho). A flushed term or an
    output below FLT_MIN is off by less than FLT_MIN each: 2^-125 absolute."""
    p, m, S, n = _softmax_fp64(ptr, s)
    a = np.abs(s.astype(F64) - m)
    eta = (1 + 4 * U) * np.exp(U * a) - 1
    deg = np.diff(ptr).astype(np.int64)
    nz = np.flatnonzero(deg)
    eta_row = np.zeros(len(deg))
    eta_row[nz] = np.maximum.reduceat(eta, ptr[:-1][nz])
    eta_max = np.repeat(eta_row, deg)
    rho = (1 + eta_max) * (1 + _gamma(13 + np.ceil(n / 256))) - 1 + n * FLT_MIN
    rel = (1 + eta) * (1 + U) / (1 - rho) - 1
    err = np.abs(got.astype(F64) - p)
    assert np.all(err <= rel * p + 2 * FLT_MIN), float(np.max(err - rel * p))


def _check_softmax_backward(ptr, p, dp, got):
    """ds = p (dp - d), d = sum p dp, with p the engine's own forward output.

    d is an FMA chain per lane (8 links), 5 butterfly adds and ceil(n / 256) tile-sum adds: at most n_B = 13 +
    ceil(n / 256) roundings per product, so |d_got - d| <= E = gamma_nB sum |p dp| + n_B 2^-126 (each operation may flush
    a subnormal result). Then ds_got = fl(p fl(dp - d_got)) = p (t + e)(1 + d1)(1 + d2) with t = dp - d, |e| <= E,
    |d1|, |d2| <= u: |ds_got - p t| <= p (gamma_2 |t| + (1 + gamma_2) E), plus 2^-125 for the two flushable results."""
    deg = np.diff(ptr).astype(np.int64)
    rows = np.repeat(np.arange(len(deg)), deg)
    p64, dp64 = p.astype(F64), dp.astype(F64)
    d = np.bincount(rows, p64 * dp64, len(deg))
    ab = np.bincount(rows, np.abs(p64 * dp64), len(deg))
    n_b = 13 + np.ceil(deg / 256)
    E = (_gamma(n_b) * ab + n_b * FLT_MIN)[rows]
    t = dp64 - d[rows]
    bound = p64 * (_gamma(2) * np.abs(t) + (1 + _gamma(2)) * E) + 2 * FLT_MIN
    err = np.abs(got.astype(F64) - p64 * t)
    assert np.all(err <= bound), float(np.max(err - bound))


def test_edge_softmax_row_length_and_stripe_boundaries():
    import softmax_oracle as SM
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    ptr = _softmax_graph(sms)
    num_v, nnz = len(ptr) - 1, int(ptr[-1])
    rng = np.random.default_rng(23)
    s = (rng.standard_normal(nnz) * 2).astype(F32)
    dp = rng.standard_normal(nnz).astype(F32)
    idx = np.zeros(nnz, np.int32)
    op = H.SpMMB200(_csr(ptr, idx), 32)          # the softmax reads ptr only: no preprocess
    s_, dp_ = torch.from_numpy(s).to(DEV), torch.from_numpy(dp).to(DEV)
    p_, ds_ = torch.full_like(s_, float("nan")), torch.full_like(s_, float("nan"))
    op.edge_softmax(s_, p_)
    op.edge_softmax_backward(p_, dp_, ds_)
    torch.cuda.synchronize()
    p, ds = p_.cpu().numpy(), ds_.cpu().numpy()
    op.close()
    assert _same(p, SM.edge_softmax_f32(ptr, s))
    assert _same(ds, SM.edge_softmax_backward_f32(ptr, p, dp))
    _check_softmax_forward(ptr, s, p)
    _check_softmax_backward(ptr, p, dp, ds)
    # the graph does reach the boundaries it is built for
    deg = np.diff(ptr)
    long_rows = np.flatnonzero(deg > 1024)
    assert long_rows.max() == num_v - 1 and np.sum(long_rows >= 4 * sms * 256) >= len(CTA_LENGTHS) + 3
    assert set(CTA_LENGTHS) <= set(deg[long_rows[long_rows >= 4 * sms * 256]].tolist())


# ---- c. autograd at the untested widths ---------------------------------------------------------------------------

def _autograd_graph(name):
    """-> (ptr, idx, b_rows)"""
    if name == "crafted":
        return _crafted()
    ptr, idx = H.gen_named_graph("c0")
    if name == "c0":
        return ptr, idx, len(ptr) - 1
    r0, r1 = 1000, 2600                        # a row block of c0: columns index all 4096 rows of B
    e0, e1 = int(ptr[r0]), int(ptr[r1])
    return H.rebase_ptr(ptr, r0, r1), idx[e0:e1].copy(), len(ptr) - 1


AUTOGRAD_GRAPHS = ["c0", "crafted", "c0_row_block"]


@pytest.mark.parametrize("graph", AUTOGRAD_GRAPHS)
@pytest.mark.parametrize("K", AUTOGRAD_WIDTHS)
def test_graph_spmm_autograd_widths(graph, K):
    import scipy.sparse as sp
    import sddmm_oracle as SO
    from oracle import cpu as O
    ptr, idx, b_rows = _autograd_graph(graph)
    M = len(ptr) - 1
    g = _csr(ptr, idx, seed=K)
    g.val.requires_grad_(True)
    b = _dense(b_rows * K, K, 3)[: b_rows * K].reshape(b_rows, K).requires_grad_(True)
    w = _dense(M * K, K, 4)[: M * K].reshape(M, K)
    mod = H.GraphSpMM(g, K, b_rows=b_rows, seg_len=32)
    c = mod(b)
    (c * w).sum().backward()
    torch.cuda.synchronize()
    c = c.detach().cpu().numpy()
    val, bn, wn = g.val.detach().cpu().numpy()[: len(idx)], b.detach().cpu().numpy(), w.cpu().numpy()
    heavy, heavy_t = _heavy_rows(mod.op), _heavy_rows(mod.transposed())
    if K % 4 == 0:                               # the vector plans split rows at seg_len 32 (the scalar one never does)
        assert len(heavy) > 0
        if graph == "crafted":
            assert len(heavy_t) > 0
    a64 = sp.csr_matrix((val.astype(F64), idx, ptr), shape=(M, b_rows))
    # forward
    whole = np.setdiff1d(np.arange(M), heavy)
    assert _bits_equal(c[whole], O.spmm_f32(ptr, idx, val, bn, K, ftz=True)[whole])
    ab = O.spmm_abssum(ptr, idx, val, bn, K)
    assert np.all(np.abs(c - a64 @ bn.astype(F64)) <= 1e-5 * ab + 1e-30)
    # dB = A^T dC
    got_db = b.grad.cpu().numpy()
    want_db, ab_t = O.spmm_t_f32(ptr, idx, val, wn, K, b_rows=b_rows, with_abs=True)
    whole_t = np.setdiff1d(np.arange(b_rows), heavy_t)
    assert _bits_equal(got_db[whole_t], want_db[whole_t])
    assert np.all(np.abs(got_db - a64.T @ wn.astype(F64)) <= 1e-5 * ab_t + 1e-30)
    # dval = sddmm(dC, B)
    got_dv = g.val.grad.cpu().numpy()[: len(idx)]
    assert _bits_equal(got_dv, SO.sddmm_f32(ptr, idx, wn, bn, K, ftz=True))
    d64, ab_v = SO.sddmm_f64(ptr, idx, wn, bn, K)
    assert np.all(np.abs(got_dv - d64) <= 1e-5 * ab_v + 1e-30)
    mod.close()


@pytest.mark.parametrize("graph", AUTOGRAD_GRAPHS)
@pytest.mark.parametrize("K", AUTOGRAD_WIDTHS)
def test_graph_attention_autograd_widths(graph, K):
    import sddmm_oracle as SO
    import softmax_oracle as SM
    from oracle import cpu as O
    from test_attention_gpu import _fp64_attention
    ptr, idx, b_rows = _autograd_graph(graph)
    M = len(ptr) - 1
    g = _csr(ptr, idx)
    mk = lambda rows, stream, grad: _dense(rows * K, 50 + K, stream)[: rows * K].reshape(rows, K).requires_grad_(grad)
    q, k, v = mk(M, 1, True), mk(b_rows, 2, True), mk(b_rows, 3, True)
    w = mk(M, 4, False)
    att = H.GraphAttention(g, K, b_rows=b_rows, seg_len=32)
    out = att(q, k, v)
    (out * w).sum().backward()
    torch.cuda.synchronize()
    qn, kn, vn, wn = (t.detach().cpu().numpy() for t in (q, k, v, w))
    got = out.detach().cpu().numpy()
    # forward: the chained oracles, bit for bit on the rows the forward plan keeps whole
    s = SO.sddmm_f32(ptr, idx, qn, kn, K, ftz=True)
    alpha = SM.edge_softmax_f32(ptr, s)
    whole = np.setdiff1d(np.arange(M), _heavy_rows(att.op))
    assert _same(got[whole], O.spmm_f32(ptr, idx, alpha, vn, K, ftz=True)[whole])
    # against fp64: forward and every gradient
    out64, (dq, dq_abs), (dk, dk_abs), (dv, dv_abs) = _fp64_attention(ptr, idx, qn, kn, vn, wn)
    assert np.all(np.abs(got - out64) <= 1e-5 * O.spmm_abssum(ptr, idx, alpha, vn, K) + 1e-30)
    for t, ref, ab in ((q, dq, dq_abs), (k, dk, dk_abs), (v, dv, dv_abs)):
        assert np.all(np.abs(t.grad.cpu().numpy() - ref) <= 1e-5 * ab + 1e-30)
    # dv = A_alpha^T dout: bit-exact on the rows the transposed plan keeps whole
    whole_t = np.setdiff1d(np.arange(b_rows), _heavy_rows(att.transposed()))
    want_dv = O.spmm_t_f32(ptr, idx, alpha, wn, K, b_rows=b_rows)
    assert _same(v.grad.cpu().numpy()[whole_t], want_dv[whole_t])
    att.close()


# ---- d. offsets past 2^31 -----------------------------------------------------------------------------------------

def _rows_of(t, rows, K):
    return t.view(-1, K)[torch.from_numpy(np.asarray(rows, np.int64)).to(DEV)].cpu().numpy()


def _check_spmm_rows(ptr, idx, val, b_dev, c_dev, K, rows, whole_rows):
    """C rows `rows` of the engine against the oracles run on the sub-problem of those rows."""
    from oracle import cpu as O
    sptr, sidx, pos, cols = _sub_problem(ptr, idx, rows)
    sval, bsub = val[pos], _rows_of(b_dev, cols, K)
    got = _rows_of(c_dev, rows, K)
    whole = np.isin(rows, whole_rows)
    assert whole.any()
    assert _bits_equal(got[whole], O.spmm_f32(sptr, sidx, sval, bsub, K, ftz=True)[whole])
    ab = O.spmm_abssum(sptr, sidx, sval, bsub, K)
    assert np.all(np.abs(got - O.spmm_f64(sptr, sidx, sval, bsub, K)) <= 1e-5 * ab + 1e-30)


def _check_sddmm_rows(ptr, idx, xr_dev, xc_dev, out_dev, K, rows):
    sptr, sidx, pos, cols = _sub_problem(ptr, idx, rows)
    got = out_dev[torch.from_numpy(pos).to(DEV)].cpu().numpy()
    _check_sddmm(sptr, sidx, _rows_of(xr_dev, rows, K), _rows_of(xc_dev, cols, K), K, got)


def test_dense_operands_past_2_31_elements():
    """num_v = 2^21 + 5 rows at K = 1024: B, C, dC and dB each hold more than 2^31 floats. Rows at the top read the top
    rows of B, and one heavy row near the end is cut into segments. run, the transposed run and sddmm are checked on
    ~4,000 sampled rows including the last 2,048."""
    import scipy.sparse as sp
    num_v, K = 2 ** 21 + 5, 1024
    dense_bytes = num_v * K * 4
    _need_memory(4 * dense_bytes + (4 << 30), host_bytes=2 << 30)
    rng = np.random.default_rng(31)
    deg = rng.integers(2, 7, num_v)
    heavy = num_v - 700
    deg[heavy] = 20_000
    ptr = np.concatenate([[0], np.cumsum(deg)]).astype(np.int32)
    rows = np.repeat(np.arange(num_v, dtype=np.int64), deg)
    cols = np.clip(rows + rng.integers(-5000, 5000, len(rows)), 0, num_v - 1)
    cols[ptr[heavy]:ptr[heavy + 1]] = rng.integers(num_v - 200_000, num_v, deg[heavy])
    cols[ptr[num_v] - 1] = num_v - 1
    idx = cols[np.lexsort((cols, rows))].astype(np.int32)
    del rows, cols
    g = _csr(ptr, idx, seed=5)
    val = g.val.cpu().numpy()
    b = _dense(num_v * K, 5, 2)
    c = torch.empty(num_v * K, device=DEV)
    op = H.SpMMB200(g, K)
    op.preprocess(b, c)
    op.run(b, c)
    dc = _dense(num_v * K, 5, 3)
    dval = torch.empty(len(idx), device=DEV)
    op.sddmm(dc, b, dval)
    torch.cuda.synchronize()
    sample = np.unique(np.concatenate([rng.choice(num_v - 2048, 2000, replace=False), np.arange(num_v - 2048, num_v)]))
    assert heavy in set(sample.tolist())
    _check_spmm_rows(ptr, idx, val, b, c, K, sample, _whole_rows(op, num_v))
    _check_sddmm_rows(ptr, idx, dc, b, dval, K, sample)
    del c, dval
    # dB = A^T dC through the transposed operator: its CSR is A^T with every column's nonzeros in CSR order
    t = op.transposed(K)
    db = torch.empty(num_v * K, device=DEV)
    t.preprocess(dc, db)
    t.run(dc, db)
    torch.cuda.synchronize()
    at = sp.csr_matrix((np.arange(len(idx), dtype=F64), idx, ptr), shape=(num_v, num_v)).T.tocsr()
    tptr, tidx, perm = at.indptr.astype(np.int32), at.indices.astype(np.int32), at.data.astype(np.int64)
    del at
    _check_spmm_rows(tptr, tidx, val[perm], dc, db, K, sample, _whole_rows(t, num_v))
    t.close()
    op.close()


def _tall_b_block(b_rows, seed=41):
    """A 48-row block whose columns spread over b_rows rows of B, the last ones included, with one row of 400."""
    rng = np.random.default_rng(seed)
    deg = rng.integers(1, 9, 48)
    deg[20] = 400
    ptr = np.concatenate([[0], np.cumsum(deg)]).astype(np.int32)
    idx = rng.integers(0, b_rows, int(ptr[-1]))
    idx[ptr[:-1]] = rng.integers(0, 16, 48)                          # every row starts low...
    idx[ptr[1:] - 1] = b_rows - 1 - rng.integers(0, 3, 48)           # ...and ends at the last rows of B
    for r in range(48):
        idx[ptr[r]:ptr[r + 1]] = np.sort(idx[ptr[r]:ptr[r + 1]])
    return ptr, idx.astype(np.int32)


@pytest.mark.parametrize("col_blocks", [1, 3])
def test_float4_offsets_up_to_the_32_bit_guard(col_blocks):
    """b_rows = 2^25 - 1 at K = 256: the last row of B starts at float4 offset 2^31 - 64, the largest B the plan accepts
    (b_rows * K / 4 <= 2^31 - 1). B (34 GB) is allocated and only the rows the block reads are written."""
    b_rows, K = 2 ** 25 - 1, 256
    _need_memory(b_rows * K * 4 + (2 << 30))
    ptr, idx = _tall_b_block(b_rows)
    M = len(ptr) - 1
    cols = np.unique(idx)
    b = torch.empty(b_rows * K, device=DEV)
    b.view(b_rows, K)[torch.from_numpy(cols.astype(np.int64)).to(DEV)] = _dense(len(cols) * K, 9, 2).view(-1, K)
    g = _csr(ptr, idx, seed=9)
    val = g.val.cpu().numpy()
    op = H.SpMMB200(g, K, b_rows=b_rows, col_blocks=col_blocks, seg_len=64)
    c = torch.full((M * K,), float("nan"), device=DEV)
    op.preprocess(b, c)
    assert op.plan_info()["n_col_blocks"] == col_blocks
    op.run(b, c)
    xr = _dense(M * K, 9, 3)
    out = torch.full((len(idx),), float("nan"), device=DEV)
    op.sddmm(xr, b, out)
    torch.cuda.synchronize()
    rows = np.arange(M)
    whole = _whole_rows(op, M)
    assert len(whole) < M                                             # the 400-nonzero row is cut into segments
    _check_spmm_rows(ptr, idx, val, b, c, K, rows, whole)
    _check_sddmm_rows(ptr, idx, xr, b, out, K, rows)
    op.close()


def test_b_past_the_32_bit_guard_is_rejected():
    """b_rows = 2^25 at K = 256 puts the last row of B at float4 offset 2^31: preprocess refuses it with EINVAL."""
    ptr, idx = _tall_b_block(2 ** 25 - 1)
    g = _csr(ptr, idx)
    op = H.SpMMB200(g, 256, b_rows=2 ** 25)
    x = torch.empty(4, device=DEV)               # never read: the plan is refused before any access to B
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    assert lib.spmm_b200_preprocess(op._h, C.c_void_p(x.data_ptr()), C.c_void_p(x.data_ptr()), stream) == -1
    assert b"32-bit" in lib.spmm_b200_last_error()
    op.close()


def test_sddmm_band_count_past_int_range():
    """64 column blocks of 33,554,433 rows: 64 * num_v + 1 > INT_MAX (band, row) segments. SDDMM walks the nonzeros
    unbanded there and must give the oracle's bits, the same as a one-block plan."""
    import sddmm_oracle as SO
    num_v, K = 33_554_433, 4
    # plan split array (65 x num_v ints) on the device and its host copy, x_row / x_col, graph arrays
    _need_memory(65 * num_v * 4 + 4 * num_v * 16 + (2 << 30), host_bytes=65 * num_v * 4 + (4 << 30))
    rng = np.random.default_rng(43)
    ptr = np.arange(num_v + 1, dtype=np.int32)
    idx = rng.integers(0, num_v, num_v).astype(np.int32)
    idx[-1] = num_v - 1
    g = _csr(ptr, idx, seed=3)
    xr, xc = _dense(num_v * K, 3, 3), _dense(num_v * K, 3, 4)
    outs = []
    for blocks in (64, 1):
        op = H.SpMMB200(g, K, col_blocks=blocks)
        op.preprocess(xc, torch.empty(num_v * K, device=DEV))
        assert op.plan_info()["n_col_blocks"] == blocks
        out = torch.full((num_v,), float("nan"), device=DEV)
        op.sddmm(xr, xc, out)
        torch.cuda.synchronize()
        outs.append(out.cpu().numpy())
        op.close()
        del out
        gc.collect()
        H.trim_memory()
    assert _bits_equal(outs[0], SO.sddmm_f32(ptr, idx, xr.cpu().numpy(), xc.cpu().numpy(), K, ftz=True))
    assert _bits_equal(outs[0], outs[1])
