"""amax / amin reduce (spmm_b200_reduce), its gradient (spmm_b200_reduce_backward) and GraphSpMM(reduce=...) on the GPU.

Bar: vout, arg, db and dval are bit-exact against the CPU restatement (tests/reduce_oracle.c, with flush-to-zero) on
every graph, width, option, partition and handle, since the winner is defined by a total order and the gradient orders
depend on K and the row lengths alone; the gradients are also within a bound on their distance to fp64 derived from
those orders. The widths launch every kernel instantiation (tests/test_reduce_oracle.py checks the list against the
dispatch table of reduce.cu).
"""
import gc

import numpy as np
import pytest

torch = pytest.importorskip("torch")

import hpc_b200 as H  # noqa: E402
import reduce_oracle as RO  # noqa: E402

HAVE_CUDA = torch.cuda.is_available()
pytestmark = [pytest.mark.gpu, pytest.mark.skipif(not HAVE_CUDA, reason="no CUDA device")]

DEV = "cuda"
F32, F64 = np.float32, np.float64
U = 2.0 ** -24
FLT_MIN = 2.0 ** -126

# reduce.cu's layout(K): float4 units at lanes 1 .. 32 with 1, 2 and 4 units per lane (4 .. 512), several 512-column
# slices (516, 1024), scalar columns at lanes 1 .. 32 in one slice (1 .. 33) and in several (515)
WIDTHS = [1, 2, 3, 7, 13, 33, 515, 4, 8, 16, 32, 64, 128, 132, 256, 260, 388, 512, 516, 1024]
BWD_WIDTHS = [3, 33, 515, 4, 32, 132, 260, 516]


@pytest.fixture(autouse=True)
def _release_memory():
    yield
    gc.collect()
    if HAVE_CUDA:
        torch.cuda.synchronize()
        torch.cuda.empty_cache()


def _bits_equal(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return a.shape == b.shape and np.array_equal(a.view(np.int32), b.view(np.int32))


def _t(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def _csr(ptr, idx, seed=7):
    nnz = len(idx)
    val = H.fill_normal(torch.empty(max(1, nnz), device=DEV), seed, 1)[:nnz] if nnz else torch.empty(0, device=DEV)
    return H.CSR(len(ptr) - 1, nnz, _t(ptr.astype(np.int32)), _t(idx.astype(np.int32)), val.contiguous())


def _dense(n, seed, stream):
    return H.fill_normal(torch.empty(max(n, 1), device=DEV), seed, stream)[:n]


def _forward(op_obj, op, vin, with_arg=True):
    M, K = op_obj.num_v, op_obj.feat_in
    vout = torch.full((max(1, M * K),), float("nan"), device=DEV)
    arg = torch.full((max(1, M * K),), -7, dtype=torch.int32, device=DEV) if with_arg else None
    op_obj.reduce(op, vin, vout, arg)
    torch.cuda.synchronize()
    return (vout[: M * K].cpu().numpy().reshape(M, K),
            arg[: M * K].cpu().numpy().reshape(M, K) if with_arg else None)


def _check_forward(ptr, idx, K, op, b_rows=None, seed=7, **opts):
    M = len(ptr) - 1
    b_rows = b_rows or M
    g = _csr(ptr, idx, seed)
    vin = _dense(b_rows * K, seed, 3)
    o = H.SpMMB200(g, K, b_rows=b_rows, **opts)
    o.preprocess(vin, torch.empty(max(1, M * K), device=DEV))
    v, a = _forward(o, op, vin)
    v2, _ = _forward(o, op, vin, with_arg=False)
    want_v, want_a = RO.reduce_f32(ptr, idx, g.val.cpu().numpy(), vin.cpu().numpy().reshape(b_rows, K), K, op)
    assert _bits_equal(v, want_v) and np.array_equal(a, want_a)
    assert _bits_equal(v2, want_v)
    info = o.plan_info()
    o.close()
    return v, info


@pytest.mark.parametrize("op", ["amax", "amin"])
@pytest.mark.parametrize("K", WIDTHS)
def test_forward_c0_every_width(K, op):
    ptr, idx = H.gen_named_graph("c0")
    _check_forward(ptr, idx, K, op)


@pytest.mark.parametrize("op,K", [("amax", 3), ("amin", 32), ("amax", 256), ("amin", 516)])
def test_forward_arxiv(op, K):
    ptr, idx = H.gen_named_graph("arxiv")
    _check_forward(ptr, idx, K, op)


@pytest.mark.parametrize("op,K", [("amax", 256), ("amin", 33)])
def test_forward_am_long_row(op, K):
    """am holds a 154 828-entry row: the CTA path."""
    ptr, idx = H.gen_named_graph("am")
    assert np.diff(ptr).max() == 154828
    _check_forward(ptr, idx, K, op)


def test_forward_reddit_full_size_sampled_rows():
    """All of reddit at K = 256 (several column blocks: one pass per band), checked on 2048 seeded rows and the longest."""
    ptr, idx = H.gen_named_graph("reddit")
    M, K = len(ptr) - 1, 256
    g = _csr(ptr, idx, 11)
    vin = _dense(M * K, 11, 3)
    o = H.SpMMB200(g, K)
    o.preprocess(vin, torch.empty(M * K, device=DEV))
    assert o.plan_info()["n_col_blocks"] > 1
    vout = torch.empty(M * K, device=DEV)
    arg = torch.empty(M * K, dtype=torch.int32, device=DEV)
    o.reduce("amax", vin, vout, arg)
    torch.cuda.synchronize()
    rng = np.random.default_rng(5)
    rows = np.unique(np.concatenate([rng.choice(M, 2048, replace=False), [int(np.argmax(np.diff(ptr)))]]))
    deg = np.diff(ptr)[rows]
    sub_ptr = np.concatenate([[0], np.cumsum(deg)]).astype(np.int32)
    pos = np.concatenate([np.arange(ptr[r], ptr[r + 1]) for r in rows]).astype(np.int64)
    val = g.val.cpu().numpy()
    want_v, want_a = RO.reduce_f32(sub_ptr, idx[pos], val[pos], vin.cpu().numpy().reshape(M, K), K, "amax")
    got_v = vout.view(M, K)[_t(rows.astype(np.int64))].cpu().numpy()
    got_a = arg.view(M, K)[_t(rows.astype(np.int64))].cpu().numpy()
    assert _bits_equal(got_v, want_v)
    sub_to_pos = np.concatenate([pos, [-1]])           # oracle positions are sub-CSR positions; -1 stays -1
    assert np.array_equal(got_a, sub_to_pos[want_a])
    o.close()


OPTION_SETS = [{}, {"col_blocks": 1}, {"col_blocks": 3}, {"reorder": 0}, {"reorder": 1}, {"row_groups": 4},
               {"col_blocks": 3, "reorder": 0}]


@pytest.mark.parametrize("K", [32, 260])
def test_same_bits_under_every_option(K):
    ptr, idx = H.gen_named_graph("arxiv")
    first = None
    for opts in OPTION_SETS:
        v, info = _check_forward(ptr, idx, K, "amax", **opts)
        if opts.get("col_blocks") == 3:
            assert info["n_col_blocks"] == 3
        first = v if first is None else first
        assert _bits_equal(v, first), opts


def _unsorted(ptr, idx, seed=5):
    rng = np.random.default_rng(seed)
    idx = idx.copy()
    for r in range(len(ptr) - 1):
        rng.shuffle(idx[ptr[r]:ptr[r + 1]])
    return idx


@pytest.mark.parametrize("K", [7, 64])
def test_unsorted_rows_and_duplicate_columns(K):
    ptr, idx = H.gen_named_graph("c0")
    idx = _unsorted(ptr, idx)
    idx[1::5] = idx[0::5][: len(idx[1::5])]          # duplicate columns inside rows
    _check_forward(ptr, idx, K, "amin")
    _check_forward(ptr, idx, K, "amax", col_blocks=3)   # unsorted rows: the plan keeps one block


@pytest.mark.parametrize("K", [32, 256])
def test_row_block(K):
    ptr, idx = H.gen_named_graph("arxiv")
    M = len(ptr) - 1
    r0, r1 = M // 3, 2 * M // 3
    lp = H.rebase_ptr(ptr, r0, r1)
    _check_forward(lp, idx[ptr[r0]:ptr[r1]], K, "amax", b_rows=M, col_blocks=3)


def _transpose_np(ptr, idx, val, b_rows):
    rows = np.repeat(np.arange(len(ptr) - 1), np.diff(ptr)).astype(np.int32)
    order = np.argsort(idx, kind="stable")
    tptr = np.concatenate([[0], np.cumsum(np.bincount(idx, minlength=b_rows))]).astype(np.int32)
    return tptr, rows[order], val[order], order


@pytest.mark.parametrize("op", ["amax", "amin"])
def test_transposed_and_column_sorted_handles(op):
    ptr, idx = H.gen_named_graph("c0")
    M, K = len(ptr) - 1, 64
    idx = _unsorted(ptr, idx)
    g = _csr(ptr, idx)
    x = _dense(M * K, 9, 3)
    o = H.SpMMB200(g, K)
    o.preprocess(x, torch.empty(M * K, device=DEV))
    val = g.val.cpu().numpy()
    xn = x.cpu().numpy().reshape(M, K)
    t = o.transposed()
    t.preprocess(x, torch.empty(M * K, device=DEV))
    v, a = _forward(t, op, x)
    tptr, tidx, tval, _ = _transpose_np(ptr, idx, val, M)
    want_v, want_a = RO.reduce_f32(tptr, tidx, tval, xn, K, op)
    assert _bits_equal(v, want_v) and np.array_equal(a, want_a)
    s = o.column_sorted()
    s.preprocess(x, torch.empty(M * K, device=DEV))
    v, a = _forward(s, op, x)
    order = np.lexsort((idx, np.repeat(np.arange(M), np.diff(ptr))))   # by row, then column, stable
    want_v, want_a = RO.reduce_f32(ptr, idx[order], val[order], xn, K, op)
    assert _bits_equal(v, want_v) and np.array_equal(a, want_a)
    s.close()
    t.close()
    o.close()


@pytest.mark.parametrize("opts", [{}, {"col_blocks": 3}])
def test_reduce_and_run_do_not_disturb_each_other(opts):
    ptr, idx = H.gen_named_graph("arxiv")
    M, K = len(ptr) - 1, 256
    g = _csr(ptr, idx)
    b = _dense(M * K, 4, 3)
    o = H.SpMMB200(g, K, **opts)
    c1, c2 = torch.empty(M * K, device=DEV), torch.empty(M * K, device=DEV)
    o.preprocess(b, c1)
    v1, a1 = _forward(o, "amax", b)
    o.run(b, c1)
    v2, a2 = _forward(o, "amax", b)
    o.run(b, c2)
    torch.cuda.synchronize()
    assert _bits_equal(v1, v2) and np.array_equal(a1, a2)
    assert torch.equal(c1.view(torch.int32), c2.view(torch.int32))
    o.close()


def test_reads_live_values():
    """reduce reads g.val as it is now, without refresh_values (run would still use the staged copy)."""
    ptr, idx = H.gen_named_graph("c0")
    M, K = len(ptr) - 1, 32
    g = _csr(ptr, idx)
    b = _dense(M * K, 4, 3)
    o = H.SpMMB200(g, K)
    o.preprocess(b, torch.empty(M * K, device=DEV))
    g.val.mul_(-2.0)
    v, a = _forward(o, "amax", b)
    want_v, want_a = RO.reduce_f32(ptr, idx, g.val.cpu().numpy(), b.cpu().numpy().reshape(M, K), K, "amax")
    assert _bits_equal(v, want_v) and np.array_equal(a, want_a)
    o.close()


def test_degenerate_inputs():
    K = 8
    for ptr in (np.zeros(6, np.int32), np.zeros(1, np.int32)):       # all rows empty (num_e = 0); no rows
        M = len(ptr) - 1
        g = _csr(ptr, np.zeros(0, np.int32))
        o = H.SpMMB200(g, K, b_rows=4)
        b = _dense(4 * K, 1, 1)
        o.preprocess(b, torch.empty(max(1, M * K), device=DEV))
        v, a = _forward(o, "amax", b)
        assert np.all(v.view(np.int32) == 0) and np.all(a == -1)
        t = o.transposed()
        db = torch.full((4 * K,), float("nan"), device=DEV)
        t.reduce_backward(torch.empty(max(1, M * K), device=DEV), torch.empty(max(1, M * K), dtype=torch.int32, device=DEV), db=db)
        torch.cuda.synchronize()
        assert torch.all(db.view(torch.int32) == 0)
        t.close()
        o.close()
    ptr, idx = H.gen_named_graph("c0")                                 # K = 0: nothing to do
    g = _csr(ptr, idx)
    o = H.SpMMB200(g, 0)
    o.preprocess(torch.empty(1, device=DEV), torch.empty(1, device=DEV))
    o.reduce("amax", torch.empty(1, device=DEV), torch.empty(1, device=DEV))
    o.close()


def test_status_codes_with_a_live_handle():
    from hpc_b200._lib import SpmmB200Error, lib
    ptr, idx = H.gen_named_graph("c0")
    M, K = len(ptr) - 1, 32
    g = _csr(ptr, idx)
    o = H.SpMMB200(g, K)
    b = _dense(M * K, 1, 1)
    o.preprocess(b, torch.empty(M * K, device=DEV))
    s = H.fill_normal(torch.empty(1, device=DEV), 1, 1)
    assert lib.spmm_b200_reduce(o._h, 1, None, s.data_ptr(), None, None) == -1          # null vin with nonzeros
    assert lib.spmm_b200_reduce(o._h, 1, b.data_ptr(), None, None, None) == -1          # null vout
    cs = o.column_sorted()
    with pytest.raises(SpmmB200Error):
        cs.reduce_backward(b, torch.empty(M * K, dtype=torch.int32, device=DEV), db=torch.empty(M * K, device=DEV))
    t = o.transposed()
    assert lib.spmm_b200_reduce_backward(t._h, b.data_ptr(), None, None, b.data_ptr(), None, None) == -1   # no arg
    assert lib.spmm_b200_reduce_backward(t._h, b.data_ptr(), b.data_ptr(), None, None, b.data_ptr(), None) == -1  # dval, no vin
    with pytest.raises(ValueError):
        o.reduce("max", b, b)
    t.close()
    cs.close()
    o.close()


# ---- backward ----------------------------------------------------------------------------------------------------

def _long_column_graph():
    """Rows of 1 .. 4 nonzeros; column 0 is in 3 * 4096 + 17 rows (CTA path, many tiles), column 1 in 2500 (warp path,
    three tiles), the rest spread over 200 columns."""
    rng = np.random.default_rng(8)
    M = 20000
    ptr, idx = [0], []
    for r in range(M):
        cols = set()
        if r < 3 * 4096 + 17:
            cols.add(0)
        if r % 7 == 0 and r // 7 < 2500:
            cols.add(1)
        for _ in range(int(rng.integers(0, 3))):
            cols.add(int(rng.integers(2, 202)))
        idx.extend(sorted(cols))
        ptr.append(len(idx))
    return np.asarray(ptr, np.int32), np.asarray(idx, np.int32), M


GRAPHS = {}


def _graph(name):
    if name not in GRAPHS:
        GRAPHS[name] = H.gen_named_graph(name) if name != "long_column" else _long_column_graph()[:2]
    return GRAPHS[name]


def _check_backward(name, K, op="amax", which=("db", "dval"), **opts):
    ptr, idx = _graph(name)
    M = len(ptr) - 1
    b_rows = int(idx.max()) + 1 if len(idx) else M
    g = _csr(ptr, idx, 13)
    b = _dense(b_rows * K, 13, 3)
    dc = _dense(M * K, 13, 4)
    o = H.SpMMB200(g, K, b_rows=b_rows, **opts)
    o.preprocess(b, torch.empty(M * K, device=DEV))
    vout = torch.empty(M * K, device=DEV)
    arg = torch.empty(M * K, dtype=torch.int32, device=DEV)
    o.reduce(op, b, vout, arg)
    t = o.transposed()
    db = torch.full((b_rows * K,), float("nan"), device=DEV) if "db" in which else None
    dval = torch.full((len(idx),), float("nan"), device=DEV) if "dval" in which else None
    t.reduce_backward(dc, arg, db=db, dval=dval, vin=b if dval is not None else None)
    torch.cuda.synchronize()
    val, bn, dcn, an = g.val.cpu().numpy(), b.cpu().numpy().reshape(b_rows, K), dc.cpu().numpy().reshape(M, K), \
        arg.cpu().numpy().reshape(M, K)
    want_db, want_dv = RO.reduce_backward_f32(ptr, idx, val, dcn, an, bn, b_rows, K, db=db is not None,
                                              dval=dval is not None)
    f64 = RO.reduce_backward_f64(ptr, idx, val, dcn, an, bn, b_rows, K)
    if db is not None:
        got = db.cpu().numpy().reshape(b_rows, K)
        assert _bits_equal(got, want_db)
        n = f64["db_terms"] + np.ceil(np.bincount(idx, minlength=b_rows) / RO.TILE)[:, None]
        gamma = n * U / (1 - n * U)
        assert np.all(np.abs(got - f64["db"]) <= gamma * f64["db_abs"] + n * FLT_MIN)
    if dval is not None:
        got = dval.cpu().numpy()
        assert _bits_equal(got, want_dv)
        n = K + 5
        assert np.all(np.abs(got - f64["dval"]) <= n * U / (1 - n * U) * f64["dval_abs"] + n * FLT_MIN)
    t.close()
    o.close()


@pytest.mark.parametrize("K", BWD_WIDTHS)
@pytest.mark.parametrize("name", ["c0", "long_column"])
def test_backward_matches_oracle(name, K):
    _check_backward(name, K)


@pytest.mark.parametrize("which", [("db",), ("dval",)])
@pytest.mark.parametrize("K", [7, 64, 516])
def test_backward_each_output_alone(K, which):
    _check_backward("long_column", K, "amin", which)


@pytest.mark.parametrize("name,K", [("arxiv", 128), ("am", 32)])
def test_backward_named_graphs(name, K):
    _check_backward(name, K, "amax", col_blocks=3 if name == "arxiv" else 0)


def test_capture_in_a_cuda_graph():
    ptr, idx = H.gen_named_graph("arxiv")
    M, K = len(ptr) - 1, 64
    g = _csr(ptr, idx)
    b, dc = _dense(M * K, 5, 3), _dense(M * K, 5, 4)
    o = H.SpMMB200(g, K, col_blocks=3)
    o.preprocess(b, torch.empty(M * K, device=DEV))
    t = o.transposed()
    outs = [(torch.empty(M * K, device=DEV), torch.empty(M * K, dtype=torch.int32, device=DEV),
             torch.empty(M * K, device=DEV), torch.empty(len(idx), device=DEV)) for _ in range(2)]

    def step(v, a, db, dval):
        o.reduce("amin", b, v, a)
        t.reduce_backward(dc, a, db=db, dval=dval, vin=b)

    step(*outs[0])
    torch.cuda.synchronize()
    for x in outs[1]:
        x.fill_(-1)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        step(*outs[1])
    graph.replay()
    torch.cuda.synchronize()
    for x, y in zip(*outs):
        assert torch.equal(x.view(torch.int32), y.view(torch.int32))
    t.close()
    o.close()


# ---- GraphSpMM(reduce=...) ---------------------------------------------------------------------------------------

@pytest.mark.parametrize("reduce", ["sum", "mean", "amax", "amin"])
@pytest.mark.parametrize("K", [7, 32])
def test_graph_spmm_reduce_matches_torch_sparse_mm(reduce, K):
    ptr, idx = H.gen_named_graph("c0")
    M = len(ptr) - 1
    g = _csr(ptr, idx, 21)
    g.val.requires_grad_(True)
    b = _dense(M * K, 21, 3).reshape(M, K).clone().requires_grad_(True)
    w = _dense(M * K, 21, 4).reshape(M, K)
    mod = H.GraphSpMM(g, K, reduce=reduce)
    c = mod(b)
    (c * w).sum().backward()
    torch.cuda.synchronize()
    tv = g.val.detach().cpu().clone().requires_grad_(True)
    tb = b.detach().cpu().clone().requires_grad_(True)
    a = torch.sparse_csr_tensor(torch.from_numpy(ptr).long(), torch.from_numpy(idx).long(), tv, size=(M, M))
    tc = torch.sparse.mm(a, tb, reduce)
    (tc * w.cpu()).sum().backward()
    assert torch.allclose(c.detach().cpu(), tc.detach(), rtol=1e-4, atol=1e-5)
    assert torch.allclose(b.grad.cpu(), tb.grad, rtol=1e-4, atol=1e-5)
    assert torch.allclose(g.val.grad.cpu(), tv.grad, rtol=1e-4, atol=1e-5)
    if reduce == "sum":
        g.val.grad = None
        b.grad = None
        plain = H.GraphSpMM(g, K)
        c2 = plain(b)
        (c2 * w).sum().backward()
        assert torch.equal(c.detach().view(torch.int32), c2.detach().view(torch.int32))
        plain.close()
    mod.close()


def test_graph_spmm_amax_follows_in_place_value_updates():
    ptr, idx = H.gen_named_graph("c0")
    M, K = len(ptr) - 1, 16
    g = _csr(ptr, idx, 22)
    b = _dense(M * K, 22, 3).reshape(M, K)
    mod = H.GraphSpMM(g, K, reduce="amax")
    mod(b)
    with torch.no_grad():
        g.val.mul_(-1.0)
    c = mod(b)
    want, _ = RO.reduce_f32(ptr, idx, g.val.detach().cpu().numpy(), b.cpu().numpy(), K, "amax")
    assert _bits_equal(c.cpu().numpy(), want)
    with pytest.raises(ValueError):
        H.GraphSpMM(g, K, reduce="max")
    mod.close()
