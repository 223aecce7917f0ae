"""Edge softmax (spmm_b200_edge_softmax / _backward) and graph attention (hpc_b200.GraphAttention) on the GPU.

Bar: both softmax kernels are bit-exact against the CPU restatement of their documented order (tests/softmax_oracle.c,
with flush-to-zero) on every graph, handle and option, since that order depends on the row length alone. NaN outputs
match as NaN (see test_edge_softmax_oracle.same_bits).
"""
import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

if not torch.cuda.is_available():
    pytest.skip("no CUDA device", allow_module_level=True)

import hpc_b200 as H  # noqa: E402
from oracle import cpu as O  # noqa: E402
import sddmm_oracle as SO  # noqa: E402
import softmax_oracle as SM  # noqa: E402

DEV = "cuda"
F32, F64 = np.float32, np.float64


def _same(a, b):
    a, b = np.asarray(a, F32), np.asarray(b, F32)
    return a.shape == b.shape and bool(np.all((np.isnan(a) & np.isnan(b)) | (a.view(np.int32) == b.view(np.int32))))


def _csr(ptr, idx):
    nnz = len(idx)
    return H.CSR(len(ptr) - 1, nnz, torch.from_numpy(np.ascontiguousarray(ptr, np.int32)).to(DEV),
                 torch.from_numpy(np.ascontiguousarray(idx, np.int32)).to(DEV),
                 H.fill_normal(torch.empty(max(nnz, 1), device=DEV), 11, 1))


def _edge_data(nnz, seed):
    rng = np.random.default_rng(seed)
    s = (rng.standard_normal(nnz) * 3).astype(F32)
    dp = rng.standard_normal(nnz).astype(F32)
    return s, dp


def _run(op, s, dp):
    """-> (p, ds) of the engine on handle op for host scores s and upstream gradient dp."""
    n = len(s)
    ds_, dp_ = torch.from_numpy(s).to(DEV), torch.from_numpy(dp).to(DEV)
    p = torch.full((max(n, 1),), float("nan"), device=DEV)
    ds = torch.full((max(n, 1),), float("nan"), device=DEV)
    op.edge_softmax(ds_, p)
    op.edge_softmax_backward(p, dp_, ds)
    torch.cuda.synchronize()
    return p[:n].cpu().numpy(), ds[:n].cpu().numpy()


def _check(ptr, s, dp, p, ds):
    want_p = SM.edge_softmax_f32(ptr, s)
    assert _same(p, want_p)
    assert _same(ds, SM.edge_softmax_backward_f32(ptr, want_p, dp))


@pytest.mark.parametrize("shape", ["c0", "arxiv", "am"])
def test_matches_oracle(shape):
    ptr, idx = H.gen_named_graph(shape)
    s, dp = _edge_data(len(idx), 1)
    op = H.SpMMB200(_csr(ptr, idx), 32)   # no preprocess: the softmax reads ptr only
    p, ds = _run(op, s, dp)
    _check(ptr, s, dp, p, ds)
    op.close()


def test_reddit_full_size():
    ptr, idx = H.gen_named_graph("reddit")
    s, dp = _edge_data(len(idx), 2)
    op = H.SpMMB200(_csr(ptr, idx), 256)
    p, ds = _run(op, s, dp)
    _check(ptr, s, dp, p, ds)
    op.close()


def _special_case():
    rng = np.random.default_rng(9)
    deg = rng.integers(0, 40, 300)
    deg[rng.random(300) < 0.25] = 0
    deg[[3, 17, 29, 40]] = [257, 1024, 1025, 5000]
    special = [9, 5, 12, 7, 300, 1, 40, 3000, 3000]   # -inf, all -inf, NaN, +inf, subnormal, single, wide; long: NaN, all -inf
    deg = np.concatenate([deg, special])
    ptr = np.concatenate([[0], np.cumsum(deg)]).astype(np.int32)
    s = (rng.standard_normal(int(ptr[-1])) * 3).astype(F32)
    row = lambda i: slice(ptr[300 + i], ptr[301 + i])
    s[row(0)][::2] = -np.inf
    s[row(1)] = -np.inf
    s[row(2)][4] = np.nan
    s[row(3)][2] = np.inf
    s[row(4)] = (rng.standard_normal(300) * 1e-39).astype(F32)
    s[row(6)] = (rng.standard_normal(40) * 40).astype(F32)
    s[row(7)][2999] = np.nan
    s[row(8)] = -np.inf
    s[ptr[40]:ptr[41]][::3] = -np.inf
    idx = rng.integers(0, len(ptr) - 1, int(ptr[-1])).astype(np.int32)
    dp = rng.standard_normal(int(ptr[-1])).astype(F32)
    dp[row(4)] *= F32(1e-36)
    return ptr, idx, s, dp


def test_edge_cases():
    ptr, idx, s, dp = _special_case()
    op = H.SpMMB200(_csr(ptr, idx), 32)
    p, ds = _run(op, s, dp)
    _check(ptr, s, dp, p, ds)
    assert np.all(p[ptr[301]:ptr[302]] == 0)                        # all -inf: zeros
    assert np.all(np.isnan(p[ptr[302]:ptr[304]]))                   # NaN / +inf: NaN rows
    assert p[ptr[305]] == 1.0
    op.close()
    for ptr0 in (np.zeros(1, np.int32), np.zeros(6, np.int32)):     # no nonzeros: nothing to do
        op = H.SpMMB200(_csr(ptr0, np.zeros(0, np.int32)), 32)
        e = torch.empty(1, device=DEV)
        op.edge_softmax(e, e)
        op.close()


@pytest.mark.parametrize("opts", [{"col_blocks": 1}, {"col_blocks": 3}, {"reorder": 0}, {"reorder": 1}])
def test_same_bits_under_options_and_repeats(opts):
    ptr, idx = H.gen_named_graph("arxiv")
    M = len(ptr) - 1
    s, dp = _edge_data(len(idx), 3)
    op = H.SpMMB200(_csr(ptr, idx), 64, **opts)
    x = torch.empty(M * 64, device=DEV)
    op.preprocess(x, torch.empty_like(x))
    p1, ds1 = _run(op, s, dp)
    p2, ds2 = _run(op, s, dp)
    _check(ptr, s, dp, p1, ds1)
    assert _same(p1, p2) and _same(ds1, ds2)
    op.close()


def test_row_blocks_equal_the_whole():
    ptr, idx = H.gen_named_graph("arxiv")
    M = len(ptr) - 1
    s, dp = _edge_data(len(idx), 4)
    op = H.SpMMB200(_csr(ptr, idx), 32)
    whole_p, whole_ds = _run(op, s, dp)
    op.close()
    bounds = H.partition_rows(ptr, 3)
    for r0, r1 in zip(bounds[:-1], bounds[1:]):
        e0, e1 = int(ptr[r0]), int(ptr[r1])
        lp = H.rebase_ptr(ptr, int(r0), int(r1))
        ob = H.SpMMB200(_csr(lp, idx[e0:e1]), 32, b_rows=M)
        p, ds = _run(ob, s[e0:e1].copy(), dp[e0:e1].copy())
        assert _same(p, whole_p[e0:e1]) and _same(ds, whole_ds[e0:e1])
        ob.close()


def test_transposed_handle_normalises_columns():
    import scipy.sparse as sp
    ptr, idx = H.gen_named_graph("arxiv")
    M, nnz = len(ptr) - 1, len(idx)
    at = sp.csr_matrix((np.arange(nnz, dtype=F64), idx, ptr), shape=(M, M)).T.tocsr()
    perm = at.data.astype(np.int64)
    s, dp = _edge_data(nnz, 5)
    op = H.SpMMB200(_csr(ptr, idx), 32)
    x = torch.empty(M * 32, device=DEV)
    op.preprocess(x, torch.empty_like(x))
    t = op.transposed()
    p, ds = _run(t, s[perm].copy(), dp[perm].copy())
    _check(at.indptr.astype(np.int32), s[perm], dp[perm], p, ds)
    t.close()
    op.close()


def test_capturable_in_a_cuda_graph():
    ptr, idx = H.gen_named_graph("arxiv")
    s, dp = _edge_data(len(idx), 6)
    op = H.SpMMB200(_csr(ptr, idx), 32)
    s_, dp_ = torch.from_numpy(s).to(DEV), torch.from_numpy(dp).to(DEV)
    p, ds = torch.full_like(s_, float("nan")), torch.full_like(s_, float("nan"))
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        op.edge_softmax(s_, p)
        op.edge_softmax_backward(p, dp_, ds)
    graph.replay()
    torch.cuda.synchronize()
    _check(ptr, s, dp, p.cpu().numpy(), ds.cpu().numpy())
    first = (p.clone(), ds.clone())
    p.fill_(float("nan"))
    ds.fill_(float("nan"))
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(p.view(torch.int32), first[0].view(torch.int32))
    assert torch.equal(ds.view(torch.int32), first[1].view(torch.int32))
    op.close()


# ---- GraphAttention ------------------------------------------------------------------------------------------------

def _dense(rows, K, seed, stream, grad=False):
    t = H.fill_normal(torch.empty(rows * K, device=DEV), seed, stream).reshape(rows, K)
    return t.requires_grad_(grad)


def _fp64_attention(ptr, idx, q, k, v, w):
    """fp64 forward and gradients of sum(w * attention(q, k, v)), with the sums of |terms| each gradient adds up."""
    import scipy.sparse as sp
    M = len(ptr) - 1
    rows = np.repeat(np.arange(M), np.diff(ptr))
    q, k, v, w = (a.astype(F64) for a in (q, k, v, w))
    s = (q[rows] * k[idx]).sum(1)
    mx = np.full(M, -np.inf)
    np.maximum.at(mx, rows, s)
    e = np.exp(s - mx[rows])
    den = np.bincount(rows, e, M)
    alpha = e / den[rows]
    A = lambda vals: sp.csr_matrix((vals, idx, ptr), shape=(M, k.shape[0]))
    out = A(alpha) @ v
    dalpha = (w[rows] * v[idx]).sum(1)
    dalpha_abs = (np.abs(w[rows]) * np.abs(v[idx])).sum(1)
    dv = A(alpha).T @ w
    dv_abs = A(alpha).T @ np.abs(w)
    d = np.bincount(rows, alpha * dalpha, M)
    ds = alpha * (dalpha - d[rows])
    ds_abs = alpha * (dalpha_abs + np.bincount(rows, alpha * dalpha_abs, M)[rows])
    dq, dq_abs = A(ds) @ k, A(ds_abs) @ np.abs(k)
    dk, dk_abs = A(ds).T @ q, A(ds_abs).T @ np.abs(q)
    return out, (dq, dq_abs), (dk, dk_abs), (dv, dv_abs)


@pytest.mark.parametrize("shape", ["c0", "arxiv"])
@pytest.mark.parametrize("K", [32, 256])
@pytest.mark.parametrize("opts", [{}, {"col_blocks": 3}], ids=["default", "col_blocks3"])
def test_graph_attention_forward_and_gradients(shape, K, opts):
    ptr, idx = H.gen_named_graph(shape)
    M = len(ptr) - 1
    g = _csr(ptr, idx)
    val0 = g.val.clone()
    q, k, v = _dense(M, K, 21, 1, True), _dense(M, K, 21, 2, True), _dense(M, K, 21, 3, True)
    w = _dense(M, K, 21, 4)
    att = H.GraphAttention(g, K, **opts)
    out = att(q, k, v)
    (out * w).sum().backward()
    torch.cuda.synchronize()
    qn, kn, vn, wn = (t.detach().cpu().numpy() for t in (q, k, v, w))
    got = out.detach().cpu().numpy()
    # forward: the chained oracles, bit for bit on the rows the forward plan keeps whole
    s = SO.sddmm_f32(ptr, idx, qn, kn, K, ftz=True)
    alpha = SM.edge_softmax_f32(ptr, s)
    want = O.spmm_f32(ptr, idx, alpha, vn, K)
    heavy = att.op.heavy_row_set()
    whole = np.asarray([r for r in range(M) if r not in heavy], np.int64)
    assert _same(got[whole], want[whole])
    ab = O.spmm_abssum(ptr, idx, alpha, vn, K)
    assert np.all(np.abs(got.astype(F64) - want) <= 1e-5 * ab + 1e-30)
    # gradients against fp64
    out64, (dq, dq_abs), (dk, dk_abs), (dv, dv_abs) = _fp64_attention(ptr, idx, qn, kn, vn, wn)
    assert np.all(np.abs(got - out64) <= 1e-5 * O.spmm_abssum(ptr, idx, alpha, vn, K) + 1e-30)
    for t, ref, ab in ((q, dq, dq_abs), (k, dk, dk_abs), (v, dv, dv_abs)):
        assert np.all(np.abs(t.grad.cpu().numpy() - ref) <= 1e-5 * ab + 1e-30)
    # dv = A_alpha^T dout: bit-exact on the rows the transposed plan keeps whole
    want_dv = O.spmm_t_f32(ptr, idx, alpha, wn, K)
    heavy_t = att.transposed().heavy_row_set()
    whole_t = np.asarray([r for r in range(M) if r not in heavy_t], np.int64)
    assert _same(v.grad.cpu().numpy()[whole_t], want_dv[whole_t])
    assert torch.equal(g.val.view(torch.int32), val0.view(torch.int32))   # g.val is never written
    att.close()


def test_gat_composition_against_dense_fp64():
    ptr, idx = H.gen_named_graph("c0")
    M, K = len(ptr) - 1, 32
    g = _csr(ptr, idx)
    h = _dense(M, K, 31, 1, True)
    a_l, a_r = _dense(K, 1, 31, 2, True), _dense(K, 1, 31, 3, True)
    w = _dense(M, K, 31, 4)
    rows = torch.repeat_interleave(torch.arange(M, device=DEV), torch.diff(g.ptr.long()))
    cols = g.idx.long()

    def gat(att_softmax, att_aggregate, h, a_l, a_r):
        el, er = (h @ a_l).squeeze(1), (h @ a_r).squeeze(1)
        e = torch.nn.functional.leaky_relu(el[rows] + er[cols], 0.2)
        return att_aggregate(att_softmax(e), h)

    att = H.GraphAttention(g, K)
    out = gat(att.softmax, att.aggregate, h, a_l, a_r)
    (out * w).sum().backward()
    grads = [t.grad.clone() for t in (h, a_l, a_r)]

    h64, al64, ar64 = (t.detach().double().requires_grad_(True) for t in (h, a_l, a_r))

    def dense_softmax(e):
        E = torch.full((M, M), float("-inf"), dtype=torch.float64, device=DEV)
        E = E.index_put((rows, cols), e)
        return torch.nan_to_num(torch.softmax(E, 1), nan=0.0)

    out64 = gat(dense_softmax, lambda P, x: P @ x, h64, al64, ar64)
    (out64 * w.double()).sum().backward()
    assert torch.allclose(out.double(), out64, rtol=1e-5, atol=1e-6)
    for got, ref in zip(grads, (h64.grad, al64.grad, ar64.grad)):
        assert torch.allclose(got.double(), ref, rtol=1e-4, atol=1e-5 * float(ref.abs().max()))
    att.close()


def test_lazy_transposed_operator_and_ownership():
    ptr, idx = H.gen_named_graph("c0")
    M, K = len(ptr) - 1, 32
    g = _csr(ptr, idx)
    val0 = g.val.clone()
    q, k, v = _dense(M, K, 41, 1), _dense(M, K, 41, 2), _dense(M, K, 41, 3)
    att = H.GraphAttention(g, K)
    att(q, k, v)
    assert att._t is None                          # no gradient needed: no transposed operator
    q.requires_grad_(True)
    att(q, k, v).sum().backward()                  # dq needs the forward operator only
    assert att._t is None and q.grad is not None
    v.requires_grad_(True)
    att(q, k, v).sum().backward()
    assert att._t is not None and v.grad is not None
    assert torch.equal(g.val.view(torch.int32), val0.view(torch.int32))
    with pytest.raises(ValueError):
        att(q.double(), k, v)
    with pytest.raises(ValueError):
        att.softmax(torch.zeros(3, device=DEV))
    att.close()
