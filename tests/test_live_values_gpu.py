"""SpMM over caller-supplied edge values: the plan option live_values and spmm_b200_run_values, on the GPU.

Bar: a live plan is the snapshot plan of the same options with each staged value replaced by the nonzero's position (on a
derived handle, its position in the source's CSR), and run_values(x) is bit-identical, on every element, to the
snapshot plan after its values are set to x and refreshed: the entries, their order and the FMA chains are the same,
only the source of the weight differs. Whole rows are also bit-exact against the CPU oracle.
"""
import ctypes as C

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

if not torch.cuda.is_available():
    pytest.skip("no CUDA device", allow_module_level=True)

import hpc_b200 as H  # noqa: E402
from hpc_b200._lib import SpmmB200Error, lib  # noqa: E402
from hpc_b200.spmm import SpMMB200  # noqa: E402
from oracle import cpu as O  # noqa: E402

DEV = "cuda"
EINVAL, ESTATE = -1, -2

# option sets that change the plan's layout: column blocks, row order, kernel variant, two-stream launches, row groups,
# host-call bands, heavy segments (small seg_len), short light tasks, several feature slices
OPTS = [{}, {"col_blocks": 3}, {"col_blocks": 5}, {"reorder": 0}, {"reorder": 1}, {"tune": 1},
        {"col_blocks": 3, "split_streams": 0}, {"col_blocks": 3, "split_streams": 1, "row_groups": 4},
        {"row_groups": 8, "reorder": 0}, {"col_blocks": 3, "host_bands": 1}, {"seg_len": 16}, {"light_steps": 16},
        {"kslice": 32}]
OPT_IDS = ["-".join(f"{k}{v}" for k, v in o.items()) or "default" for o in OPTS]
KS = [0, 4, 8, 32, 64, 128, 256, 512, 36, 6]   # 36 and 6: the scalar kernel (K % 4 != 0)

_GRAPHS = {}


def _graph(shape="c0"):
    if shape not in _GRAPHS:
        _GRAPHS[shape] = H.gen_named_graph(shape)
    return _GRAPHS[shape]


def _dev(a, dt):
    return torch.from_numpy(np.ascontiguousarray(a, dt)).to(DEV)


def _csr(ptr, idx, val=None):
    nnz = len(idx)
    v = torch.zeros(max(nnz, 1), device=DEV) if val is None else val
    return H.CSR(len(ptr) - 1, nnz, _dev(ptr, np.int32), _dev(idx, np.int32), v)


def _positions(n):
    """arange(n) reinterpreted as float32 bits: a snapshot plan staging these holds the live plan's .y words."""
    return torch.arange(max(n, 1), dtype=torch.int32, device=DEV).view(torch.float32)


def _values(n, seed, special=False):
    rng = np.random.default_rng(seed)
    x = rng.standard_normal(max(n, 1)).astype(np.float32)
    if special:   # NaN, +-inf and subnormals sprinkled in
        pick = rng.choice(len(x), size=min(len(x), 40), replace=False)
        for j, p in enumerate(pick):
            x[p] = (np.nan, np.inf, -np.inf, np.float32(1e-40), np.float32(-3e-39))[j % 5]
    return x


def _bits(t):
    return t.contiguous().view(torch.int32)


def _same(a, b):
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    return a.shape == b.shape and bool(np.all((np.isnan(a) & np.isnan(b)) | (a.view(np.int32) == b.view(np.int32))))


def _dense(rows, K, seed):
    return H.fill_normal(torch.empty((rows, K), device=DEV), seed, 5)


def _shuffle_rows(ptr, idx, seed):
    """The same matrix with the nonzeros of every row in a random order (a CSR that is not column-sorted)."""
    rng = np.random.default_rng(seed)
    out = idx.copy()
    for r in range(len(ptr) - 1):
        out[ptr[r]:ptr[r + 1]] = rng.permutation(out[ptr[r]:ptr[r + 1]])
    return out


def _row_block(ptr, idx, r0, r1):
    return (ptr[r0:r1 + 1] - ptr[r0]).astype(np.int32), idx[ptr[r0]:ptr[r1]].copy()


class Pair:
    """A live operator and a snapshot operator with the same options over the same pattern. kind: "plain" (the CSR,
    b_rows > num_v for a row block), "transposed" or "sorted" (derived from a source over the pattern)."""

    def __init__(self, ptr, idx, K, opts, kind="plain", b_rows=0, snap_val=None):
        self.K, self.kind = K, kind
        self.g_live = _csr(ptr, idx, torch.from_numpy(_values(len(idx), 99)).to(DEV))
        self.g_snap = _csr(ptr, idx, snap_val)
        if kind == "plain":
            self.src = None
            self.live = SpMMB200(self.g_live, K, b_rows=b_rows, live_values=1, **opts)
            self.snap = SpMMB200(self.g_snap, K, b_rows=b_rows, **opts)
        else:
            self.src = (SpMMB200(self.g_live, K, b_rows=b_rows), SpMMB200(self.g_snap, K, b_rows=b_rows))
            make = "transposed" if kind == "transposed" else "column_sorted"
            self.live = getattr(self.src[0], make)(K, live_values=1, **opts)
            self.snap = getattr(self.src[1], make)(K, **opts)
        self.rows_in, self.rows_out = self.live.b_rows, self.live.num_v
        for op in (self.live, self.snap):
            op.preprocess(torch.empty(max(self.rows_in * K, 1), device=DEV), torch.empty(max(self.rows_out * K, 1), device=DEV))

    def snapshot_run(self, x, b):
        """Option 0: values set to x, refreshed, run."""
        self.g_snap.val[: len(x)].copy_(x)
        self.snap.refresh_values()
        out = torch.full((self.rows_out, self.K), float("nan"), device=DEV)
        self.snap.run(b, out)
        return out

    def live_run(self, x, b):
        out = torch.full((self.rows_out, self.K), float("nan"), device=DEV)
        self.live.run_values(x, b, out)
        return out

    def close(self):
        for op in (self.live, self.snap) + (self.src or ()):
            op.close()


# ---- 1. plan identity --------------------------------------------------------------------------------------------

def _plans_equal(a, b):
    nb = a.plan_info(0)["n_col_blocks"]
    assert nb == b.plan_info(0)["n_col_blocks"]
    for blk in range(nb):
        assert a.plan_info(blk) == b.plan_info(blk)
        pa, pb = a.plan_arrays(blk), b.plan_arrays(blk)
        for name in pa:
            assert np.array_equal(pa[name], pb[name]), (blk, name)
    return nb


@pytest.mark.parametrize("opts", OPTS, ids=OPT_IDS)
@pytest.mark.parametrize("K", [32, 256, 36])
def test_plan_is_the_snapshot_plan_of_positions(K, opts):
    ptr, idx = _graph()
    pair = Pair(ptr, idx, K, opts, snap_val=_positions(len(idx)))
    nb = _plans_equal(pair.live, pair.snap)
    if opts.get("col_blocks", 1) > 1 and K % 4 == 0:
        assert nb == opts["col_blocks"]
    if K % 4 == 0:   # the .y words are the CSR positions
        arrs = pair.live.plan_arrays(0)
        lp = arrs["lpanel"]
        nz = lp[:, 0] >= 0
        assert nz.any() and np.all((lp[nz, 1] >= 0) & (lp[nz, 1] < len(idx)))
    pair.close()


@pytest.mark.parametrize("opts", [{}, {"col_blocks": 3, "seg_len": 16}, {"reorder": 0, "row_groups": 4}, {"kslice": 32}],
                         ids=["default", "cb3-seg16", "natural-rg4", "kslice32"])
@pytest.mark.parametrize("kind", ["transposed", "sorted"])
def test_derived_plan_stages_source_positions(kind, opts):
    ptr, idx = _graph()
    if kind == "sorted":
        idx = _shuffle_rows(ptr, idx, 5)
    pair = Pair(ptr, idx, 64, opts, kind=kind, snap_val=_positions(len(idx)))
    _plans_equal(pair.live, pair.snap)
    # and those words are a permutation of the source's positions
    ys = []
    for blk in range(pair.live.plan_info(0)["n_col_blocks"]):
        a = pair.live.plan_arrays(blk)
        ys += [a["lpanel"][a["lpanel"][:, 0] >= 0, 1], a["panel"][a["panel"][:, 0] >= 0, 1]]
    assert np.array_equal(np.sort(np.concatenate(ys)), np.arange(len(idx)))
    pair.close()


# ---- 2. bits against the snapshot and the oracle -----------------------------------------------------------------

def _check_oracle_rows(pair, ptr, idx, x, b, got, K):
    """Whole rows of the live result bit-exact against the CPU oracle with values x."""
    if K == 0:
        return
    xs, bs = x.cpu().numpy()[: len(idx)], b.cpu().numpy()
    if pair.kind == "transposed":
        ref = O.spmm_t_f32(ptr, idx, xs, bs, K, b_rows=pair.rows_out, ftz=True).reshape(pair.rows_out, K)
    elif pair.kind == "sorted":
        rows = np.repeat(np.arange(len(ptr) - 1), np.diff(ptr))
        perm = np.lexsort((idx, rows))   # stable: the sorted operator's order
        ref = O.spmm_f32(ptr, idx[perm], xs[perm], bs, K, ftz=True).reshape(pair.rows_out, K)
    else:
        ref = O.spmm_f32(ptr, idx, xs, bs, K, ftz=True).reshape(pair.rows_out, K)
    heavy = pair.live.heavy_row_set() if K % 4 == 0 else set()
    whole = np.asarray([r for r in range(pair.rows_out) if r not in heavy], np.int64)
    assert len(whole) > 0
    assert _same(got.cpu().numpy()[whole], ref[whole])


def _bits_case(pair, ptr, idx, K, seed, special=False):
    x = torch.from_numpy(_values(len(idx), seed, special)).to(DEV)
    b = _dense(pair.rows_in, K, seed)
    want = pair.snapshot_run(x, b)
    got = pair.live_run(x, b)
    torch.cuda.synchronize()
    assert torch.equal(_bits(got), _bits(want))
    _check_oracle_rows(pair, ptr, idx, x, b, got, K)


@pytest.mark.parametrize("special", [False, True], ids=["finite", "nan-inf-subnormal"])
@pytest.mark.parametrize("opts", OPTS, ids=OPT_IDS)
@pytest.mark.parametrize("K", KS)
def test_run_values_equals_refreshed_snapshot(K, opts, special):
    ptr, idx = _graph()
    pair = Pair(ptr, idx, K, opts)
    _bits_case(pair, ptr, idx, K, seed=K + 1, special=special)
    pair.close()


DERIVED_OPTS = [{}, {"col_blocks": 3, "seg_len": 16}, {"col_blocks": 3, "split_streams": 1, "row_groups": 4}]


@pytest.mark.parametrize("special", [False, True], ids=["finite", "nan-inf-subnormal"])
@pytest.mark.parametrize("opts", DERIVED_OPTS, ids=["default", "cb3-seg16", "cb3-two-streams"])
@pytest.mark.parametrize("K", [4, 32, 64, 256, 36])
@pytest.mark.parametrize("kind", ["block", "transposed", "sorted"])
def test_run_values_on_row_blocks_and_derived_handles(kind, K, opts, special):
    ptr, idx = _graph()
    b_rows = 0
    if kind == "block":   # rows [1000, 2600) of c0: columns index the whole B
        b_rows = len(ptr) - 1
        ptr, idx = _row_block(ptr, idx, 1000, 2600)
    elif kind == "sorted":
        idx = _shuffle_rows(ptr, idx, 7)
    pair = Pair(ptr, idx, K, opts, kind="plain" if kind == "block" else kind, b_rows=b_rows)
    _bits_case(pair, ptr, idx, K, seed=3 * K + 2, special=special)
    pair.close()


# ---- 3. live reads -----------------------------------------------------------------------------------------------

@pytest.mark.parametrize("K,opts", [(32, {}), (256, {"col_blocks": 3}), (36, {})])
def test_run_reads_the_current_values(K, opts):
    ptr, idx = _graph()
    pair = Pair(ptr, idx, K, opts)
    b = _dense(pair.rows_in, K, 4)
    out = torch.empty((pair.rows_out, K), device=DEV)
    x1 = torch.from_numpy(_values(len(idx), 1)).to(DEV)
    x2 = torch.from_numpy(_values(len(idx), 2)).to(DEV)
    pair.g_live.val.copy_(x1)
    pair.live.run(b, out)                       # no refresh_values: run reads g.val now
    r1 = out.clone()
    pair.g_live.val.copy_(x2)
    pair.live.run(b, out)
    r2 = out.clone()
    assert torch.equal(_bits(r1), _bits(pair.snapshot_run(x1, b)))
    assert torch.equal(_bits(r2), _bits(pair.snapshot_run(x2, b)))
    # two value arrays back to back on one stream, each giving its own result
    o1, o2 = pair.live_run(x1, b), pair.live_run(x2, b)
    assert torch.equal(_bits(o1), _bits(r1)) and torch.equal(_bits(o2), _bits(r2))
    # run -> run_values -> run, repeated: every repeat gives the same bits
    for _ in range(3):
        pair.live.run(b, out)
        assert torch.equal(_bits(out), _bits(r2))
        assert torch.equal(_bits(pair.live_run(x1, b)), _bits(r1))
    pair.close()


def test_transposed_run_reads_the_source_values():
    ptr, idx = _graph()
    pair = Pair(ptr, idx, 64, {"col_blocks": 3}, kind="transposed")
    x = torch.from_numpy(_values(len(idx), 8)).to(DEV)
    b = _dense(pair.rows_in, 64, 8)
    pair.g_live.val.copy_(x)   # the source operator's values, in its CSR positions
    out = torch.empty((pair.rows_out, 64), device=DEV)
    pair.live.run(b, out)
    assert torch.equal(_bits(out), _bits(pair.snapshot_run(x, b)))
    pair.close()


def test_refresh_values_after_idx_changes():
    """refresh_values on a live plan re-stages idx (and the positions): needed after idx changes, not after val does."""
    ptr, idx = _graph()
    pair = Pair(ptr, idx, 32, {})
    idx2 = _shuffle_rows(ptr, idx, 3)   # same rows, other order: one column block, same row lengths
    pair.g_live.idx.copy_(_dev(idx2, np.int32))
    pair.g_snap.idx.copy_(_dev(idx2, np.int32))
    pair.live.refresh_values()
    x = torch.from_numpy(_values(len(idx), 9)).to(DEV)
    b = _dense(pair.rows_in, 32, 9)
    assert torch.equal(_bits(pair.live_run(x, b)), _bits(pair.snapshot_run(x, b)))
    pair.close()


# ---- 4. full size ------------------------------------------------------------------------------------------------

def test_reddit_k256_full_size():
    ptr, idx = _graph("reddit")
    K = 256
    pair = Pair(ptr, idx, K, {})
    assert pair.live.plan_info(0)["n_col_blocks"] == 5
    x = H.fill_normal(torch.empty(len(idx), device=DEV), 7, 3)
    b = H.fill_normal(torch.empty(pair.rows_in * K, device=DEV), 7, 4).reshape(pair.rows_in, K)
    want = pair.snapshot_run(x, b)
    got = pair.live_run(x, b)
    assert pair.live.launches_per_run == 10   # five column blocks, two launches each (two streams)
    torch.cuda.synchronize()
    assert torch.equal(_bits(got), _bits(want))
    pair.close()


# ---- 5. CUDA graph -----------------------------------------------------------------------------------------------

@pytest.mark.parametrize("K,opts", [(64, {"col_blocks": 3, "split_streams": 1, "row_groups": 4}), (36, {})])
def test_cuda_graph_replay_reads_new_values(K, opts):
    ptr, idx = _graph()
    pair = Pair(ptr, idx, K, opts)
    x = torch.from_numpy(_values(len(idx), 10)).to(DEV)
    x2 = torch.from_numpy(_values(len(idx), 11)).to(DEV)
    b = _dense(pair.rows_in, K, 10)
    out = torch.empty((pair.rows_out, K), device=DEV)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        pair.live.run_values(x, b, out)   # warm-up outside the capture
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        pair.live.run_values(x, b, out)
    x.copy_(x2)
    out.fill_(float("nan"))
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(_bits(out), _bits(pair.snapshot_run(x2, b)))
    pair.close()


# ---- 6. stacked layers and host calls ----------------------------------------------------------------------------

@pytest.mark.parametrize("opts", [{}, {"col_blocks": 3}, {"col_blocks": 3, "host_bands": 1}])
def test_run_host_and_gather_on_a_live_plan(opts):
    ptr, idx = _graph()
    K = 64
    pair = Pair(ptr, idx, K, opts)
    b = _dense(pair.rows_in, K, 12)
    dev_out = torch.empty((pair.rows_out, K), device=DEV)
    pair.live.run(b, dev_out)
    h_out = torch.full((pair.rows_out, K), float("nan")).pin_memory()
    pair.live.run_host(b.cpu().pin_memory(), h_out)
    assert torch.equal(_bits(h_out), _bits(dev_out.cpu()))
    # stacked-layer epilogue: final rows also go to the target at a row offset
    x = torch.from_numpy(_values(len(idx), 12)).to(DEV)
    tgt = torch.full((pair.rows_out + 8, K), float("nan"), device=DEV)
    pair.live.set_gather([tgt], 8)
    got = pair.live_run(x, b)
    pair.live.set_gather([], 0)
    torch.cuda.synchronize()
    assert torch.equal(_bits(tgt[8:]), _bits(got))
    assert torch.equal(_bits(got), _bits(pair.snapshot_run(x, b)))
    pair.close()


# ---- 7. errors ---------------------------------------------------------------------------------------------------

def _code(fn):
    with pytest.raises(SpmmB200Error) as e:
        fn()
    return e.value.code, str(e.value)


def test_errors():
    ptr, idx = _graph()
    K = 32
    g = _csr(ptr, idx, torch.from_numpy(_values(len(idx), 1)).to(DEV))
    M = g.num_v
    b, out, x = _dense(M, K, 1), torch.empty((M, K), device=DEV), torch.from_numpy(_values(len(idx), 2)).to(DEV)
    snap = SpMMB200(g, K)
    snap.preprocess(b, out)
    code, msg = _code(lambda: snap.run_values(x, b, out))
    assert code == ESTATE and "live_values" in msg
    live = SpMMB200(g, K, live_values=1)
    code, msg = _code(lambda: live.run_values(x, b, out))   # no preprocess
    assert code == ESTATE and "preprocess" in msg
    live.preprocess(b, out)
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    assert lib.spmm_b200_run_values(live._h, None, C.c_void_p(b.data_ptr()), C.c_void_p(out.data_ptr()), st) == EINVAL
    assert _code(lambda: live.set_option("live_values", 2))[0] == EINVAL
    assert _code(lambda: live.set_option("live_values", -1))[0] == EINVAL
    # switching the option invalidates the plan
    live.set_option("live_values", 0)
    assert _code(lambda: live.run(b, out))[0] == ESTATE
    with pytest.raises(ValueError):   # the Python check: val shorter than num_e
        snap.run_values(x[:10], b, out)
    live.close()
    snap.close()


# ---- 8. graph attention without staging --------------------------------------------------------------------------

def _staged_attention(ptr, idx, q, k, v, w, opts):
    """The attention step composed from snapshot operators, staging the values before every run."""
    K = q.shape[1]
    buf = torch.zeros(len(idx), device=DEV)
    op = SpMMB200(_csr(ptr, idx, buf), K, **opts)
    op.preprocess(torch.empty_like(k), torch.empty_like(q))
    t = op.transposed(K)
    t.preprocess(torch.empty_like(q), torch.empty_like(k))

    def run(o, vals, b, rows):
        buf.copy_(vals)
        o.refresh_values()
        c = torch.empty((rows, K), device=DEV)
        o.run(b, c)
        return c

    s, p = torch.empty(len(idx), device=DEV), torch.empty(len(idx), device=DEV)
    op.sddmm(q, k, s)
    op.edge_softmax(s, p)
    out = run(op, p, v, q.shape[0])
    dalpha, ds = torch.empty_like(p), torch.empty_like(p)
    op.sddmm(w, v, dalpha)
    dv = run(t, p, w, k.shape[0])
    op.edge_softmax_backward(p, dalpha, ds)
    dq = run(op, ds, k, q.shape[0])
    dk = run(t, ds, q, k.shape[0])
    torch.cuda.synchronize()
    t.close()
    op.close()
    return out, dq, dk, dv


@pytest.mark.parametrize("shape,K,opts", [("c0", 32, {}), ("c0", 64, {"col_blocks": 3, "seg_len": 16}), ("arxiv", 256, {})])
def test_attention_never_restages(shape, K, opts, monkeypatch):
    ptr, idx = _graph(shape)
    M = len(ptr) - 1
    q, k, v, w = (H.fill_normal(torch.empty(M * K, device=DEV), 21, i).reshape(M, K) for i in range(4))
    want = _staged_attention(ptr, idx, q, k, v, w, opts)

    def refuse(self):
        raise AssertionError("GraphAttention must not restage values")

    monkeypatch.setattr(SpMMB200, "refresh_values", refuse)
    g = _csr(ptr, idx, torch.full((len(idx),), 7.0, device=DEV))
    val0 = g.val.clone()
    att = H.GraphAttention(g, K, **opts)
    qg, kg, vg = (x.clone().requires_grad_(True) for x in (q, k, v))
    out = att(qg, kg, vg)
    (out * w).sum().backward()
    torch.cuda.synchronize()
    for got, exp in zip((out.detach(), qg.grad, kg.grad, vg.grad), want):
        assert torch.equal(_bits(got), _bits(exp))
    assert torch.equal(g.val, val0)   # g.val is never written
    att.close()
