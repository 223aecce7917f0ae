"""SDDMM (spmm_b200_sddmm) and the differentiable SpMM (hpc_b200.GraphSpMM) on the GPU.

Bar: sddmm is bit-exact against the CPU restatement of its documented order (tests/sddmm_oracle.c, with flush-to-zero)
on every graph, option and partition, since that order depends on K alone.
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

DEV = "cuda"


def _csr(ptr, idx, val=None, seed=7):
    M, nnz = len(ptr) - 1, len(idx)
    d_val = (H.fill_normal(torch.empty(nnz, device=DEV), seed, 1) if val is None
             else torch.from_numpy(np.ascontiguousarray(val, np.float32)).to(DEV))
    return H.CSR(M, nnz, torch.from_numpy(np.ascontiguousarray(ptr, np.int32)).to(DEV),
                 torch.from_numpy(np.ascontiguousarray(idx, np.int32)).to(DEV), d_val)


def _dense(n, seed, stream):
    return H.fill_normal(torch.empty(max(n, 0), device=DEV), seed, stream)


def _sddmm(ptr, idx, K, b_rows=None, seed=7, **opts):
    """-> (engine out, oracle out) for x_row = N(0, .1) num_v x K, x_col = N(0, .1) b_rows x K."""
    M = len(ptr) - 1
    b_rows = b_rows or M
    g = _csr(ptr, idx, seed=seed)
    xr, xc = _dense(M * K, seed, 3), _dense(b_rows * K, seed, 4)
    op = H.SpMMB200(g, K, b_rows=b_rows, **opts)
    op.preprocess(xc, torch.empty(max(1, M * K), device=DEV))
    out = torch.full((max(1, len(idx)),), float("nan"), device=DEV)
    op.sddmm(xr, xc, out)
    torch.cuda.synchronize()
    got = out[: len(idx)].cpu().numpy()
    want = SO.sddmm_f32(ptr, idx, xr.cpu().numpy(), xc.cpu().numpy(), K, ftz=True)
    op.close()
    return got, want


def _bits_equal(a, b):
    return a.shape == b.shape and np.array_equal(a.view(np.int32), b.view(np.int32))


@pytest.mark.parametrize("shape", ["c0", "arxiv"])
@pytest.mark.parametrize("K", [0, 4, 32, 33, 64, 256, 512, 8, 128, 1024])
def test_matches_oracle(shape, K):
    ptr, idx = H.gen_named_graph(shape)
    got, want = _sddmm(ptr, idx, K)
    assert _bits_equal(got, want)
    if K == 0:
        assert np.all(got.view(np.int32) == 0)


def _edge_cases():
    rng = np.random.default_rng(5)
    out = {"empty_graph": (np.zeros(1, np.int32), np.zeros(0, np.int32)),
           "nnz_zero": (np.zeros(6, np.int32), np.zeros(0, np.int32))}
    ptr = np.array([0, 0, 5000, 5000, 5003], np.int32)               # one row far longer than seg_len
    out["long_row"] = (ptr, np.sort(rng.integers(0, 4, 5003)).astype(np.int32))
    deg = np.full(64, 300)                                               # every row heavy
    ptr = np.concatenate([[0], np.cumsum(deg)]).astype(np.int32)
    out["all_heavy"] = (ptr, np.sort(rng.integers(0, 64, (64, 300)), axis=1).ravel().astype(np.int32))
    ptr = np.array([0, 4, 4, 9], np.int32)
    out["duplicates"] = (ptr, np.array([1, 1, 1, 2, 0, 0, 2, 2, 2], np.int32))
    p2, i2 = H.gen_named_graph("c0")
    i2 = i2.copy()
    for r in range(len(p2) - 1):                                         # unsorted rows
        rng.shuffle(i2[p2[r]:p2[r + 1]])
    out["unsorted"] = (p2, i2)
    return out


EDGE = _edge_cases()


@pytest.mark.parametrize("name", sorted(EDGE))
@pytest.mark.parametrize("K", [4, 32, 33, 256])
def test_edge_cases(name, K):
    ptr, idx = EDGE[name]
    opts = {"seg_len": 64} if name == "all_heavy" else {}
    got, want = _sddmm(ptr, idx, K, **opts)
    assert _bits_equal(got, want)


OPTION_SETS = [{}, {"col_blocks": 1}, {"col_blocks": 3}, {"reorder": 0}, {"reorder": 1}, {"seg_len": 64},
               {"kslice": 32}, {"split_streams": 0, "col_blocks": 3},
               {"split_streams": 1, "col_blocks": 3}, {"host_bands": 1, "col_blocks": 4}]


@pytest.mark.parametrize("K", [32, 256], ids=["K32", "K256"])
def test_same_bits_under_every_option(K):
    ptr, idx = H.gen_named_graph("arxiv")
    first = None
    for opts in OPTION_SETS:
        got, want = _sddmm(ptr, idx, K, **opts)
        assert _bits_equal(got, want), opts
        first = got if first is None else first
        assert _bits_equal(got, first), opts


def test_column_blocks_are_in_effect():
    """The band-major path is exercised: col_blocks = 3 gives a three-block plan on arxiv."""
    ptr, idx = H.gen_named_graph("arxiv")
    g = _csr(ptr, idx)
    x = _dense((len(ptr) - 1) * 64, 1, 1)
    op = H.SpMMB200(g, 64, col_blocks=3)
    op.preprocess(x, torch.empty_like(x))
    assert op.plan_info()["n_col_blocks"] == 3
    op.close()


@pytest.mark.parametrize("K", [32, 256])
def test_row_blocks_concatenate_to_the_whole(K):
    ptr, idx = H.gen_named_graph("arxiv")
    M = len(ptr) - 1
    g = _csr(ptr, idx)
    xr, xc = _dense(M * K, 9, 3), _dense(M * K, 9, 4)
    whole = torch.empty(len(idx), device=DEV)
    op = H.SpMMB200(g, K)
    op.preprocess(xc, torch.empty(M * K, device=DEV))
    op.sddmm(xr, xc, whole)
    parts = []
    bounds = H.partition_rows(ptr, 3)
    for r0, r1 in zip(bounds[:-1], bounds[1:]):
        e0, e1 = int(ptr[r0]), int(ptr[r1])
        lp = H.rebase_ptr(ptr, int(r0), int(r1))
        gb = H.CSR(int(r1 - r0), e1 - e0, torch.from_numpy(lp).to(DEV), g.idx[e0:e1].contiguous(), g.val[e0:e1].contiguous())
        ob = H.SpMMB200(gb, K, b_rows=M)
        ob.preprocess(xc, torch.empty(max(1, (r1 - r0) * K), device=DEV))
        o = torch.empty(max(1, e1 - e0), device=DEV)
        ob.sddmm(xr[r0 * K: r1 * K].contiguous(), xc, o)
        torch.cuda.synchronize()
        parts.append(o[: e1 - e0].cpu().numpy())
        ob.close()
    torch.cuda.synchronize()
    assert _bits_equal(np.concatenate(parts), whole.cpu().numpy())
    op.close()


def test_reddit_k256_full_size():
    """All 114.6 M outputs of the reddit shape at K = 256 (column blocks: the band-major launch) against the oracle."""
    ptr, idx = H.gen_named_graph("reddit")
    got, want = _sddmm(ptr, idx, 256)
    assert _bits_equal(got, want)


def test_identity_with_the_forward_product():
    """sum_e val[e] * sddmm(dC, B)[e] == <dC, A·B> (both are sum over nonzeros and columns of val * dC * B)."""
    ptr, idx = H.gen_named_graph("c0")
    M, K = len(ptr) - 1, 64
    g = _csr(ptr, idx)
    b, dc = _dense(M * K, 3, 3), _dense(M * K, 3, 4)
    c = torch.empty(M * K, device=DEV)
    dval = torch.empty(len(idx), device=DEV)
    op = H.SpMMB200(g, K)
    op.preprocess(b, c)
    op.run(b, c)
    op.sddmm(dc, b, dval)
    torch.cuda.synchronize()
    lhs = float((g.val.double() * dval.double()).sum())
    rhs = float((dc.double() * c.double()).sum())
    _, ab = SO.sddmm_f64(ptr, idx, dc.cpu().numpy(), b.cpu().numpy(), K)
    scale = float((np.abs(g.val.cpu().numpy().astype(np.float64)) * ab).sum())
    assert abs(lhs - rhs) <= 1e-6 * scale
    op.close()


@pytest.mark.parametrize("opts", [{}, {"col_blocks": 3}])
def test_run_sddmm_run_and_repeat_are_bit_identical(opts):
    ptr, idx = H.gen_named_graph("arxiv")
    M, K = len(ptr) - 1, 256
    g = _csr(ptr, idx)
    b, dc = _dense(M * K, 4, 3), _dense(M * K, 4, 4)
    c1, c2 = torch.empty(M * K, device=DEV), torch.empty(M * K, device=DEV)
    o1, o2 = torch.empty(len(idx), device=DEV), torch.empty(len(idx), device=DEV)
    op = H.SpMMB200(g, K, **opts)
    op.preprocess(b, c1)
    op.run(b, c1)
    op.sddmm(dc, b, o1)
    op.run(b, c2)
    op.sddmm(dc, b, o2)
    torch.cuda.synchronize()
    assert torch.equal(c1.view(torch.int32), c2.view(torch.int32))
    assert torch.equal(o1.view(torch.int32), o2.view(torch.int32))
    op.close()


@pytest.mark.parametrize("opts", [{}, {"col_blocks": 3}])
def test_sddmm_is_capturable_in_a_cuda_graph(opts):
    ptr, idx = H.gen_named_graph("arxiv")
    M, K = len(ptr) - 1, 64
    g = _csr(ptr, idx)
    b, dc = _dense(M * K, 5, 3), _dense(M * K, 5, 4)
    ref, out = torch.empty(len(idx), device=DEV), torch.full((len(idx),), float("nan"), device=DEV)
    op = H.SpMMB200(g, K, **opts)
    op.preprocess(b, torch.empty(M * K, device=DEV))
    op.sddmm(dc, b, ref)                 # warm-up: sets up the band prefix outside the capture
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        op.sddmm(dc, b, out)
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(out.view(torch.int32), ref.view(torch.int32))
    op.close()


# ---- GraphSpMM ---------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("shape", ["c0", "arxiv"])
@pytest.mark.parametrize("K", [32, 256])
def test_graph_spmm_gradients(shape, K):
    ptr, idx = H.gen_named_graph(shape)
    M = len(ptr) - 1
    g = _csr(ptr, idx)
    g.val.requires_grad_(True)
    b = _dense(M * K, 6, 3).reshape(M, K).requires_grad_(True)
    w = _dense(M * K, 6, 4).reshape(M, K)
    mod = H.GraphSpMM(g, K)

    def step():
        b.grad = None
        g.val.grad = None
        c = mod(b)
        (c * w).sum().backward()
        torch.cuda.synchronize()
        return c.detach().cpu().numpy()

    c = step()
    val = g.val.detach().cpu().numpy()
    bn, wn = b.detach().cpu().numpy(), w.cpu().numpy()
    # forward: the operator's own run
    light = mod.op.plan_arrays()["row_perm"]
    fwd = O.spmm_f32(ptr, idx, val, bn, K)
    assert _bits_equal(c[light], fwd[light])
    # dB = A^T dC (dC = w): bit-exact on the rows A^T keeps whole, within tolerance on the others and against fp64
    want_db, ab = O.spmm_t_f32(ptr, idx, val, wn, K, with_abs=True)
    got_db = b.grad.cpu().numpy()
    heavy = mod.transposed().heavy_row_set()
    whole = np.asarray([r for r in range(M) if r not in heavy], np.int64)
    assert _bits_equal(got_db[whole], want_db[whole])
    assert np.all(np.abs(got_db.astype(np.float64) - want_db) <= 1e-5 * ab + 1e-30)
    import scipy.sparse as sp
    a64 = sp.csr_matrix((val.astype(np.float64), idx, ptr), shape=(M, M))
    assert np.all(np.abs(got_db - a64.T @ wn.astype(np.float64)) <= 1e-5 * ab + 1e-30)
    # dval = sddmm(dC, B)
    got_dv = g.val.grad.cpu().numpy()
    assert _bits_equal(got_dv, SO.sddmm_f32(ptr, idx, wn, bn, K, ftz=True))
    d64, ab64 = SO.sddmm_f64(ptr, idx, wn, bn, K)
    assert np.all(np.abs(got_dv - d64) <= 1e-5 * ab64 + 1e-30)
    # an optimizer-style in-place update of the edge values is picked up by the next forward and backward
    with torch.no_grad():
        g.val.mul_(0.5)
    c = step()
    val = g.val.detach().cpu().numpy()
    assert _bits_equal(c[light], O.spmm_f32(ptr, idx, val, bn, K)[light])
    want_db = O.spmm_t_f32(ptr, idx, val, wn, K)
    assert _bits_equal(b.grad.cpu().numpy()[whole], want_db[whole])
    assert _bits_equal(g.val.grad.cpu().numpy(), SO.sddmm_f32(ptr, idx, wn, bn, K, ftz=True))
    mod.close()


def test_graph_spmm_gradient_only_where_needed():
    """No transposed operator is built when B needs no gradient, and dval is None when val needs none."""
    ptr, idx = H.gen_named_graph("c0")
    M, K = len(ptr) - 1, 32
    g = _csr(ptr, idx)
    g.val.requires_grad_(True)
    b = _dense(M * K, 8, 3).reshape(M, K)
    mod = H.GraphSpMM(g, K)
    mod(b).sum().backward()
    assert mod._t is None and g.val.grad is not None
    g.val.requires_grad_(False)
    b.requires_grad_(True)
    mod(b).sum().backward()
    assert b.grad is not None and mod._t is not None
    mod.close()
