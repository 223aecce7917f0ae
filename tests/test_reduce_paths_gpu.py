"""amax / amin reduce and its gradient on every kernel path, at the inputs where a comparison-decided kernel goes wrong.

reduce.cu promises a total order (NaN above every number; larger or smaller value; equal values, -0 == +0 included, to
the smaller CSR position), so its bits cannot depend on how a row is split over lane groups, warps, CTAs or column-block
passes. The tests here make ties the common case (values from small sets whose products are exact in fp32) and sprinkle
NaN, infinities, overflow to inf, 0 * inf, subnormals and -0 into them, then run:

  a/b. the forward on c0 (warp kernel) and on a graph built around the row-length and stripe thresholds (CTA kernel,
       stripes past the long-row launch's first grid, rows that live in the last column band only), at widths that
       reach every lane count and (W, VEC) instantiation, with 1, 3 and 5 column blocks and with and without arg;
  c.   the backward on columns of A at the tile, warp / CTA and worker-round boundaries, with duplicate columns,
       non-finite dC on empty rows and +inf on losing columns;
  d.   both past 2^31 elements;
  e.   the alignment rule and 4-byte-offset buffers.

Bar: vout, db and dval bit-equal to the CPU restatement (tests/reduce_oracle.c, flush-to-zero) with NaN matching NaN
(payload and sign are not part of the contract), arg equal, every output's 64-element guard tail untouched, and on
finite data the fp64 bound of tests/test_reduce_gpu.py. Each test also asserts that its inputs reach the cases it is
built for. The thresholds are read from the sources; tests/test_reduce_oracle.py checks without a device that the widths
and lengths below reach each side of them.
"""
import collections
import gc
import os
import re

import numpy as np
import pytest

torch = pytest.importorskip("torch")

import hpc_b200 as H  # noqa: E402
import reduce_oracle as RO  # noqa: E402
from hpc_b200._lib import lib  # noqa: E402
from test_kernel_paths_gpu import _csr, _need_memory, _rows_of, _same, _sub_problem  # noqa: E402

HAVE_CUDA = torch.cuda.is_available()
pytestmark = [pytest.mark.gpu, pytest.mark.skipif(not HAVE_CUDA, reason="no CUDA device")]

DEV = "cuda"
F32, F64 = np.float32, np.float64
U = 2.0 ** -24
FLT_MIN = 2.0 ** -126
CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "hpc_b200", "csrc")


def source_constants():
    """The namespace-scope integer constexprs of rows.cuh and reduce.cu (kRowBlock, kRowWarps, kWarpMax, kTile,
    kBwdWarpMax, ...)."""
    env = {}
    for name in ("rows.cuh", "reduce.cu"):
        src = open(os.path.join(CSRC, name)).read()
        for k, expr in re.findall(r"^constexpr\s+(?:int|long long)\s+(k\w+)\s*=\s*([^;]+);", src, re.M):
            env[k] = int(eval(expr.replace("/", "//"), {}, dict(env)))
    return env


SRC = source_constants()
K_WARP_MAX, K_TILE, K_BWD_WARP_MAX = SRC["kWarpMax"], SRC["kTile"], SRC["kBwdWarpMax"]
K_ROW_BLOCK, K_ROW_WARPS = SRC["kRowBlock"], SRC["kRowWarps"]

# forward: float4 at lanes 1 .. 32 with 1, 2 and 4 units per lane (4 .. 512), 512-column slices (516, 1024), scalar
# columns at lanes 1, 4 and 32 in one slice (1, 3, 33) and in several (515)
FWD_WIDTHS = [1, 3, 4, 8, 16, 32, 33, 64, 128, 256, 512, 515, 516, 1024]
# each side of the warp / CTA threshold, and a few long rows up to ~70,000
FWD_ROW_LENGTHS = [K_WARP_MAX - 1, K_WARP_MAX, K_WARP_MAX + 1, 2 * K_WARP_MAX + 1, 8 * K_WARP_MAX + 1, 70_000]

# backward: lane groups of L = 1 (K = 1, 4), 4 (3, 16), 8 (32) and 32 (33, 128, 516; 516 spans two slices)
BWD_WIDTHS = [1, 3, 4, 16, 32, 33, 128, 516]


def bwd_workers(lanes):
    """Lane groups of the backward CTA kernel: tiles per round."""
    return K_ROW_WARPS * 32 // lanes


# Columns of A (rows of Aᵀ): each side of a tile and of the warp / CTA threshold, exactly one round of 8 workers, and
# past one round at every worker count, ending partway through the last round
BWD_COLUMN_LENGTHS = ([K_TILE - 1, K_TILE, K_TILE + 1, K_BWD_WARP_MAX, K_BWD_WARP_MAX + 1, bwd_workers(32) * K_TILE]
                      + [(bwd_workers(lanes) + 1) * K_TILE + 5 for lanes in (32, 8, 4)] + [300_000])

GUARD = 64
SENTINEL = 0x7FA5A5A5   # a NaN bit pattern the kernels never produce (the GPU's NaN is 0x7FFFFFFF)


@pytest.fixture(autouse=True)
def _release_memory():
    yield
    gc.collect()
    if HAVE_CUDA:
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        H.trim_memory()


# ---- helpers -----------------------------------------------------------------------------------------------------

def _guarded(n, dtype=torch.float32, lead=0):
    """n elements of dtype after `lead` sentinel elements, followed by GUARD sentinel elements -> (buffer, view)."""
    buf = torch.full((lead + n + GUARD,), SENTINEL, dtype=torch.int32, device=DEV)
    view = buf[lead:lead + n]
    return buf, view if dtype == torch.int32 else view.view(torch.float32)


def _untouched(buf, lead, n):
    b = buf.view(torch.int32)
    return bool(torch.all(b[:lead] == SENTINEL)) and bool(torch.all(b[lead + n:] == SENTINEL))


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def _bits_equal_dev(a, b):
    return torch.equal(a.view(torch.int32), b.view(torch.int32))


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


# ---- tie-heavy inputs with non-finite values ----------------------------------------------------------------------

B_SET = np.array([0.0, -0.0, 0.5, -0.5, 1.0, -1.0, 1.5, -1.5, 2.0, -2.0], F32)
VAL_SET = np.array([0.5, -0.5, 1.0, -1.0, 2.0, -2.0], F32)
SUBNORMAL = F32(2.0 ** -130)


def _sprinkle(rng, a, rate, values):
    """Set about rate * a.size elements of a (flat) to values drawn from `values`."""
    n = rng.binomial(a.size, rate)
    a.reshape(-1)[rng.integers(0, a.size, n)] = rng.choice(np.asarray(values, F32), n)


def _tie_values(rng, idx, b_rows, K, positive_val=False, specials=True):
    """val[nnz] and vin[b_rows, K]: B from {±0, ±0.5, ±1, ±1.5, ±2}, val from {±0.5, ±1, ±2} (every product exact),
    with NaN in both, ±inf, 2^40 in B against 2^100 in val (overflow to +inf), ±0 in val against ±inf (NaN), and
    subnormal B (flushed to a signed zero)."""
    nnz = len(idx)
    vals = VAL_SET[VAL_SET > 0] if positive_val else VAL_SET
    val = vals[rng.integers(0, len(vals), nnz)]
    vin = B_SET[rng.integers(0, len(B_SET), (b_rows, K), dtype=np.int8)]
    _sprinkle(rng, vin, 1e-2, [SUBNORMAL, -SUBNORMAL])
    if specials:
        _sprinkle(rng, vin, 1e-4, [np.nan])
        _sprinkle(rng, vin, 2e-4, [np.inf, -np.inf])
        _sprinkle(rng, vin, 3e-4, [2.0 ** 40])
        _sprinkle(rng, val, 2e-4, [np.nan])
        _sprinkle(rng, val, 2e-4, [2.0 ** 100])
        _sprinkle(rng, val, 1e-3, [0.0, -0.0])
        # planted: 0 * inf and 2^100 * 2^40 in every input
        for e in rng.integers(0, nnz, 32):
            val[e], vin[idx[e], rng.integers(0, K)] = rng.choice([0.0, -0.0]), rng.choice([np.inf, -np.inf])
        for e in rng.integers(0, nnz, 32):
            val[e], vin[idx[e], rng.integers(0, K)] = 2.0 ** 100, 2.0 ** 40
    return val, vin


def _messages(val, vin, pos, idx, cols):
    """fl(val[e] * vin[idx[e], j]) for e in pos, j < cols, as the flush-to-zero build computes it (no product of the
    values above is subnormal, so flushing the inputs is enough)."""
    b = vin[idx[pos], :cols]
    b = np.where(np.abs(b) < FLT_MIN, np.copysign(F32(0), b), b)
    with np.errstate(all="ignore"):
        return val[pos][:, None] * b


def _forward_reach(ptr, idx, val, vin, vout, arg, rows, band_of_pos=None, cols=16):
    """Counts, over rows `rows` and columns j < cols, of outputs whose winning value (NaN matching NaN, -0 == +0) sits at
    two or more positions — by the warp or CTA kind of row — of NaN winners with a later NaN in CTA rows, of ties in
    rows spanning several bands and of winners with an equal value in a later band. Asserts that the winner is never
    the last equal position, so that a reversed tie rule would show."""
    n_cols = min(cols, vin.shape[1])
    st = collections.Counter()
    for r in rows:
        pos = np.arange(ptr[r], ptr[r + 1])
        if not len(pos):
            continue
        m = _messages(val, vin, pos, idx, n_cols)
        w, a = vout[r, :n_cols], arg[r, :n_cols]
        eq = (m == w) | (np.isnan(m) & np.isnan(w))
        tie = eq.sum(0) >= 2
        last = pos[len(pos) - 1 - np.argmax(eq[::-1], 0)]
        assert np.all(last[tie] != a[tie])
        kind = "cta" if len(pos) > K_WARP_MAX else "warp"
        st[kind + "_tie"] += int(tie.sum())
        st[kind + "_finite_tie"] += int((tie & np.isfinite(w)).sum())
        st[kind + "_nan_tie"] += int((tie & np.isnan(w)).sum())
        if band_of_pos is not None:
            bands = band_of_pos[pos]
            if bands[0] != bands[-1]:
                st["multiband_tie"] += int(tie.sum())
            st["combine_equal"] += int((eq & (bands[:, None] > band_of_pos[a][None, :])).any(0).sum())
    return st


# ---- a/b. forward ------------------------------------------------------------------------------------------------

def _boundary_graph(sms, seed=17):
    """-> (ptr, idx, b_rows, special rows). Rows of 0..8 nonzeros, and FWD_ROW_LENGTHS placed in the first grid of the
    long-row launch (4 * SMs CTAs of kRowBlock-row stripes) and beyond it; two long rows in one 32-row ballot group in
    the first grid and beyond it; long rows at the first row past the grid and at num_v - 1; and a long and a short row
    whose columns all lie in the top 2,000 rows of B, that is, in the last column band. Columns ascend in every row,
    with duplicates."""
    first = 4 * sms * K_ROW_BLOCK
    num_v = max(160_000, first + 12_288)
    b_rows = num_v
    rng = np.random.default_rng(seed)
    deg = rng.integers(0, 9, num_v)
    deg[rng.random(num_v) < 0.2] = 0
    for i, n in enumerate(FWD_ROW_LENGTHS):
        deg[1000 + 37 * i] = n                           # first grid
        deg[first + 3000 + 41 * i] = n                   # beyond it
    deg[[64_000, 64_005]] = [K_WARP_MAX + 1, 8 * K_WARP_MAX + 1]     # one ballot group, first grid
    deg[[first + 6400, first + 6401]] = [70_000, K_WARP_MAX + 1]     # one ballot group, beyond it
    deg[first] = K_WARP_MAX + 1
    deg[num_v - 1] = 8 * K_WARP_MAX + 1
    last_band_rows = [30_000, 30_001]
    deg[last_band_rows] = [2 * K_WARP_MAX + 3, 40]
    ptr = np.concatenate([[0], np.cumsum(deg)]).astype(np.int32)
    idx = rng.integers(0, b_rows, int(ptr[-1])).astype(np.int32)
    for r in last_band_rows:
        idx[ptr[r]:ptr[r + 1]] = rng.integers(b_rows - 2000, b_rows, deg[r])
    rows = np.repeat(np.arange(num_v), deg)
    idx = idx[np.lexsort((idx, rows))]
    return ptr, idx, b_rows, np.asarray(last_band_rows)


GRAPHS = {}


def _fwd_graph(name):
    if name not in GRAPHS:
        if name == "c0":
            ptr, idx = H.gen_named_graph("c0")
            GRAPHS[name] = (ptr, idx, len(ptr) - 1, np.zeros(0, np.int64))
        else:
            GRAPHS[name] = _boundary_graph(_sms())
    return GRAPHS[name]


def _reduce_guarded(o, op, vin, with_arg=True):
    n = o.num_v * o.feat_in
    vb, vout = _guarded(n)
    ab, arg = _guarded(n, torch.int32) if with_arg else (None, None)
    o.reduce(op, vin, vout, arg)
    torch.cuda.synchronize()
    assert _untouched(vb, 0, n) and (ab is None or _untouched(ab, 0, n))
    return vout, arg


@pytest.mark.parametrize("K", FWD_WIDTHS)
@pytest.mark.parametrize("graph", ["c0", "boundary"])
def test_forward_ties_and_non_finite_on_every_path(graph, K):
    ptr, idx, b_rows, last_band_rows = _fwd_graph(graph)
    M = len(ptr) - 1
    deg = np.diff(ptr)
    rng = np.random.default_rng(1000 + K)
    val, vin = _tie_values(rng, idx, b_rows, K)
    if len(last_band_rows):
        # the rows of the last band only: every message negative, NaN or -inf, so that under amax a winner wrongly
        # combined with band 0's +0 placeholder shows
        top = vin[b_rows - 2000:]
        vin[b_rows - 2000:] = np.where(np.abs(top) < FLT_MIN, F32(0.5), np.abs(top))
        for r in last_band_rows:
            val[ptr[r]:ptr[r + 1]] = -VAL_SET[rng.integers(0, 3, deg[r]) * 2]
    g = _csr(ptr, idx, val)
    vin_d = _dev(vin.reshape(-1))
    sample = np.unique(np.concatenate([rng.choice(M, min(M, 3000), replace=False), np.flatnonzero(deg > K_WARP_MAX),
                                       last_band_rows]))
    blocks = (1, 3, 5) if K % 4 == 0 else (1,)
    for op in ("amax", "amin"):
        want_v, want_a = RO.reduce_f32(ptr, idx, val, vin, K, op)
        first = None
        for nb in blocks:
            o = H.SpMMB200(g, K, b_rows=b_rows, col_blocks=nb)
            o.preprocess(vin_d, torch.empty(M * K, device=DEV))
            assert o.plan_info()["n_col_blocks"] == nb
            begins = np.asarray([o.plan_info(b)["col_begin"] for b in range(nb)])
            vout, arg = _reduce_guarded(o, op, vin_d)
            vout2, _ = _reduce_guarded(o, op, vin_d, with_arg=False)
            o.close()
            assert _bits_equal_dev(vout, vout2), (op, nb)
            if first is None:
                first = (vout, arg)
                got_v, got_a = vout.cpu().numpy().reshape(M, K), arg.cpu().numpy().reshape(M, K)
                assert _same(got_v, want_v), op
                assert np.array_equal(got_a, want_a), op
            else:
                assert _bits_equal_dev(vout, first[0]) and torch.equal(arg, first[1]), (op, nb)
            del vout, vout2, arg
            # the inputs reach the cases they are built for (on the oracle's result, which the GPU's equals)
            band_of_pos = np.searchsorted(begins, idx, "right") - 1 if nb > 1 else None
            st = _forward_reach(ptr, idx, val, vin, want_v, want_a, sample, band_of_pos)
            assert st["warp_tie"] >= 100 and st["warp_finite_tie"] >= 50, st
            if graph == "boundary":
                assert st["cta_tie"] >= 5 and st["cta_finite_tie"] >= 1 and st["cta_nan_tie"] >= 1, st
            if nb > 1:
                assert st["multiband_tie"] >= 20 and st["combine_equal"] >= 1, st
                for r in last_band_rows:              # band 0 is empty for them: the empty-row store runs first
                    assert begins[-1] <= idx[ptr[r]]
        if graph == "boundary" and op == "amax":
            assert np.any(want_v[last_band_rows] < 0)
        del first


def test_boundary_graph_reaches_the_stripes():
    """The forward graph places long rows where the long-row launch's stripe loop and ballots can go wrong."""
    sms = _sms()
    ptr, idx, b_rows, last_band_rows = _fwd_graph("boundary")
    num_v, first = len(ptr) - 1, 4 * sms * K_ROW_BLOCK
    deg = np.diff(ptr)
    long_rows = np.flatnonzero(deg > K_WARP_MAX)
    assert long_rows.max() == num_v - 1 and first in set(long_rows.tolist())
    assert set(FWD_ROW_LENGTHS) <= set(deg[:first].tolist()) and set(FWD_ROW_LENGTHS) <= set(deg[first:].tolist())
    groups = long_rows // 32
    shared = groups[1:][groups[1:] == groups[:-1]] * 32
    assert np.any(shared < first) and np.any(shared >= first)
    for r in last_band_rows:
        assert idx[ptr[r]] >= b_rows - 2000
    assert deg[last_band_rows].max() > K_WARP_MAX and deg[last_band_rows].min() <= K_WARP_MAX


# ---- c. backward -------------------------------------------------------------------------------------------------

def _bwd_graph(sms, seed=29):
    """-> (ptr, idx, b_rows, empty rows of A). 310,000 rows of A, every tenth left empty; the others hold 0..4 random
    columns and are drawn (with replacement, so rows hold duplicate columns) into columns of BWD_COLUMN_LENGTHS
    entries, each length placed once in the long-row launch's first grid of Aᵀ rows and once beyond it."""
    first = 4 * sms * K_ROW_BLOCK
    b_rows = first + 12_288
    num_v = 310_000
    rng = np.random.default_rng(seed)
    empty = np.flatnonzero(np.arange(num_v) % 10 == 7)
    live = np.setdiff1d(np.arange(num_v), empty)
    long_cols = np.asarray([c for i in range(len(BWD_COLUMN_LENGTHS)) for c in (500 + 37 * i, first + 3000 + 41 * i)])
    deg = rng.integers(0, 5, len(live))
    rows = [np.repeat(live, deg)]
    base = rng.integers(0, b_rows, len(rows[0]))
    base[np.isin(base, long_cols)] += 1                  # keeps the long columns at their exact lengths
    cols = [base]
    for i, n in enumerate(BWD_COLUMN_LENGTHS):
        for c in long_cols[2 * i:2 * i + 2]:
            rows.append(rng.choice(live, n))
            cols.append(np.full(n, c))
    rows, cols = np.concatenate(rows), np.concatenate(cols)
    order = np.lexsort((cols, rows))
    ptr = np.concatenate([[0], np.cumsum(np.bincount(rows, minlength=num_v))]).astype(np.int32)
    return ptr, cols[order].astype(np.int32), b_rows, empty


def _fp64_bounds_hold(ptr, idx, val, dcn, an, bn, b_rows, K, got_db, got_dv):
    """tests/test_reduce_gpu.py's bound, where the fp64 result is finite."""
    f64 = RO.reduce_backward_f64(ptr, idx, val, dcn, an, bn, b_rows, K)
    ok = True
    with np.errstate(invalid="ignore"):                  # inf - inf where the fp64 result is not finite (masked out)
        if got_db is not None:
            n = f64["db_terms"] + np.ceil(np.bincount(idx, minlength=b_rows) / RO.TILE)[:, None]
            err = np.abs(got_db - f64["db"]) - (n * U / (1 - n * U) * f64["db_abs"] + n * FLT_MIN)
            ok &= bool(np.all(err[np.isfinite(f64["db"])] <= 0))
        if got_dv is not None:
            n = K + 5
            err = np.abs(got_dv - f64["dval"]) - (n * U / (1 - n * U) * f64["dval_abs"] + n * FLT_MIN)
            ok &= bool(np.all(err[np.isfinite(f64["dval"])] <= 0))
    return ok


@pytest.mark.parametrize("variant", ["ties", "inf_loses"])
@pytest.mark.parametrize("K", BWD_WIDTHS)
def test_backward_tiles_rounds_and_non_finite(K, variant):
    """db and dval alone and together. ties: amax over tie-heavy finite values with duplicate columns. inf_loses: amin
    with val > 0 and +inf in B, which loses, so dval must skip it rather than multiply it by a zero mask. In both, dC
    holds NaN and ±inf on the empty rows of A (arg == -1), which nothing may read."""
    if "bwd" not in GRAPHS:
        GRAPHS["bwd"] = _bwd_graph(_sms())
    ptr, idx, b_rows, empty = GRAPHS["bwd"]
    M, nnz = len(ptr) - 1, len(idx)
    rng = np.random.default_rng(2000 + K)
    op = "amax" if variant == "ties" else "amin"
    val, vin = _tie_values(rng, idx, b_rows, K, positive_val=variant == "inf_loses", specials=False)
    if variant == "inf_loses":
        _sprinkle(rng, vin, 2e-3, [np.inf])
    dcn = rng.standard_normal((M, K)).astype(F32)
    dcn[empty] = np.where(np.arange(len(empty))[:, None] % 2 == 0, F32(np.nan), F32(np.inf))
    dcn[empty[1::4]] = -np.inf
    g = _csr(ptr, idx, val)
    vin_d, dc_d = _dev(vin.reshape(-1)), _dev(dcn.reshape(-1))
    o = H.SpMMB200(g, K, b_rows=b_rows)
    o.preprocess(vin_d, torch.empty(M * K, device=DEV))
    _, arg = _reduce_guarded(o, op, vin_d)
    an = arg.cpu().numpy().reshape(M, K)
    t = o.transposed()
    want_db, want_dv = RO.reduce_backward_f32(ptr, idx, val, dcn, an, vin, b_rows, K)
    for which in (("db",), ("dval",), ("db", "dval")):
        dbb, db = _guarded(b_rows * K) if "db" in which else (None, None)
        dvb, dval = _guarded(nnz) if "dval" in which else (None, None)
        t.reduce_backward(dc_d, arg, db=db, dval=dval, vin=vin_d if dval is not None else None)
        torch.cuda.synchronize()
        got_db = db.cpu().numpy().reshape(b_rows, K) if db is not None else None
        got_dv = dval.cpu().numpy() if dval is not None else None
        if db is not None:
            assert _untouched(dbb, 0, b_rows * K) and _same(got_db, want_db), which
        if dval is not None:
            assert _untouched(dvb, 0, nnz) and _same(got_dv, want_dv), which
        if which == ("db", "dval"):
            assert _fp64_bounds_hold(ptr, idx, val, dcn, an, vin, b_rows, K, got_db, got_dv)
    t.close()
    o.close()
    # the inputs reach the cases they are built for
    assert np.all(an[empty] == -1) and np.all(np.isfinite(want_db))     # dC's NaN / inf on empty rows reach no db
    rows = np.repeat(np.arange(M), np.diff(ptr))
    dup = np.zeros(nnz, bool)
    same = (idx[1:] == idx[:-1]) & (rows[1:] == rows[:-1])
    dup[1:] |= same
    dup[:-1] |= same
    won = an[an >= 0]
    assert np.count_nonzero(dup[won]) >= 100              # winners that are one of several duplicate entries
    if variant == "ties":
        assert np.all(np.isfinite(want_dv))
    else:
        inf_cols = np.isinf(vin).any(1)[idx]              # entries whose column of B holds +inf somewhere
        assert np.count_nonzero(inf_cols & np.isfinite(want_dv)) >= 10


def test_backward_graph_reaches_the_thresholds():
    sms = _sms()
    if "bwd" not in GRAPHS:
        GRAPHS["bwd"] = _bwd_graph(sms)
    ptr, idx, b_rows, _ = GRAPHS["bwd"]
    first = 4 * sms * K_ROW_BLOCK
    lengths = np.bincount(idx, minlength=b_rows)
    for n in BWD_COLUMN_LENGTHS:
        at = np.flatnonzero(lengths == n)
        assert np.any(at < first) and np.any(at >= first), n
    assert b_rows > first


# ---- d. offsets past 2^31 elements -------------------------------------------------------------------------------

def test_offsets_past_2_31_elements():
    """num_v = 2^21 + 5 rows at K = 1024 (two 512-column slices): vin, vout, arg, dC and dB each hold more than 2^31
    elements. One heavy row near the end takes the CTA kernel and columns reach the last rows of B. The forward is
    checked on ~4,000 sampled rows, the last 2,048 included; db on sampled columns of B, the last ones included, and
    dval on all their entries, through the sub-problem of those columns (positions outside it renumbered to -1, which
    changes neither)."""
    num_v, K = 2 ** 21 + 5, 1024
    dense = num_v * K * 4
    _need_memory(5 * dense + (4 << 30), host_bytes=4 << 30)
    rng = np.random.default_rng(37)
    deg = rng.integers(2, 7, num_v)
    heavy = num_v - 700
    deg[heavy] = 20_000
    ptr = np.concatenate([[0], np.cumsum(deg)]).astype(np.int32)
    rows = np.repeat(np.arange(num_v, dtype=np.int64), deg)
    cols = np.clip(rows + rng.integers(-5000, 5000, len(rows)), 0, num_v - 1)
    cols[ptr[heavy]:ptr[heavy + 1]] = rng.integers(num_v - 200_000, num_v, deg[heavy])
    cols[ptr[num_v] - 1] = num_v - 1
    idx = cols[np.lexsort((cols, rows))].astype(np.int32)
    del cols
    g = _csr(ptr, idx, seed=5)
    val = g.val.cpu().numpy()[: len(idx)]
    vin = H.fill_normal(torch.empty(num_v * K, device=DEV), 5, 2)
    o = H.SpMMB200(g, K)
    o.preprocess(vin, vin)                        # preprocess reads neither buffer
    vout_b, vout = _guarded(num_v * K)
    arg_b, arg = _guarded(num_v * K, torch.int32)
    o.reduce("amax", vin, vout, arg)
    torch.cuda.synchronize()
    assert _untouched(vout_b, 0, num_v * K) and _untouched(arg_b, 0, num_v * K)
    sample = np.unique(np.concatenate([rng.choice(num_v - 2048, 2000, replace=False), np.arange(num_v - 2048, num_v)]))
    assert heavy in set(sample.tolist())
    sptr, sidx, pos, scols = _sub_problem(ptr, idx, sample)
    want_v, want_a = RO.reduce_f32(sptr, sidx, val[pos], _rows_of(vin, scols, K), K, "amax")
    assert _same(_rows_of(vout, sample, K), want_v)
    assert np.array_equal(_rows_of(arg, sample, K), np.concatenate([pos, [-1]])[want_a])
    del vout, vout_b
    # backward on the transposed operator
    dc = H.fill_normal(torch.empty(num_v * K, device=DEV), 5, 3)
    t = o.transposed()
    db_b, db = _guarded(num_v * K)
    dv_b, dval = _guarded(len(idx))
    t.reduce_backward(dc, arg, db=db, dval=dval, vin=vin)
    torch.cuda.synchronize()
    assert _untouched(db_b, 0, num_v * K) and _untouched(dv_b, 0, len(idx))
    bcols = np.unique(np.concatenate([rng.choice(num_v - 2048, 2000, replace=False), np.arange(num_v - 2048, num_v)]))
    epos = np.flatnonzero(np.isin(idx, bcols))           # every entry of those columns, in CSR order
    erows = rows[epos]
    arows = np.unique(erows)                             # the rows of A (dC, arg) they read
    sptr = np.concatenate([[0], np.cumsum(np.bincount(np.searchsorted(arows, erows), minlength=len(arows)))])
    sidx = np.searchsorted(bcols, idx[epos])
    a_full = _rows_of(arg, arows, K)
    k = np.clip(np.searchsorted(epos, a_full), 0, len(epos) - 1)
    a_sub = np.where(epos[k] == a_full, k, -1)
    dcs, vins = _rows_of(dc, arows, K), _rows_of(vin, bcols, K)
    want_db, want_dv = RO.reduce_backward_f32(sptr, sidx, val[epos], dcs, a_sub, vins, len(bcols), K)
    got_db = _rows_of(db, bcols, K)
    got_dv = dval[_dev(epos)].cpu().numpy()
    assert _same(got_db, want_db) and _same(got_dv, want_dv)
    assert _fp64_bounds_hold(sptr, sidx, val[epos], dcs, a_sub, vins, len(bcols), K, got_db, got_dv)
    assert np.count_nonzero(a_sub >= 0) > 1000 and np.bincount(sidx).max() > K_TILE
    t.close()
    o.close()


# ---- e. alignment and bounds -------------------------------------------------------------------------------------

def test_misaligned_buffers_are_refused_when_k_is_a_multiple_of_4():
    """K % 4 == 0 reads and writes float4 / int4: every one of vin, vout, arg (forward) and dc, arg, vin, db (backward)
    must be 16-byte aligned, and a misaligned one is refused with SPMM_B200_EINVAL before anything is written."""
    ptr, idx = H.gen_named_graph("c0")
    M, K = len(ptr) - 1, 32
    g = _csr(ptr, idx)
    n = M * K
    vin = H.fill_normal(torch.empty(n + 4, device=DEV), 3, 3)
    o = H.SpMMB200(g, K)
    o.preprocess(vin, torch.empty(n, device=DEV))
    t = o.transposed()
    vb, vout = _guarded(n + 4)
    ab, arg = _guarded(n + 4, torch.int32)
    db_b, db = _guarded(n + 4)
    ptrs = {"vin": vin.data_ptr(), "vout": vout.data_ptr(), "arg": arg.data_ptr()}
    for name in ptrs:
        p = dict(ptrs, **{name: ptrs[name] + 4})
        assert lib.spmm_b200_reduce(o._h, 1, p["vin"], p["vout"], p["arg"], None) == -1, name
        assert b"16-byte aligned" in lib.spmm_b200_last_error(), name
    torch.cuda.synchronize()
    assert _untouched(vb, 0, 0) and _untouched(ab, 0, 0)
    o.reduce("amax", vin, vout[:n], arg[:n])         # a valid call, for the backward's arg
    ptrs = {"dc": vin.data_ptr(), "arg": arg.data_ptr(), "vin": vin.data_ptr(), "db": db.data_ptr()}
    for name in ptrs:
        p = dict(ptrs, **{name: ptrs[name] + 4})
        assert lib.spmm_b200_reduce_backward(t._h, p["dc"], p["arg"], p["vin"], p["db"], None, None) == -1, name
        assert b"16-byte aligned" in lib.spmm_b200_last_error(), name
    torch.cuda.synchronize()
    assert _untouched(db_b, 0, 0)
    t.close()
    o.close()


@pytest.mark.parametrize("K", [3, 33, 515])
def test_odd_widths_take_any_float_alignment(K):
    """K % 4 != 0 reads and writes single floats: every buffer 4 bytes past a 16-byte boundary, with guards of sentinel
    elements before and after each output, gives the oracle's bits on tie-heavy, non-finite data."""
    ptr, idx = H.gen_named_graph("c0")
    M, nnz = len(ptr) - 1, len(idx)
    rng = np.random.default_rng(3000 + K)
    val, vin = _tie_values(rng, idx, M, K)
    dcn = rng.standard_normal((M, K)).astype(F32)
    lead = GUARD + 1
    g = _csr(ptr, idx, val)
    ins = {}
    for name, a in (("vin", vin), ("dc", dcn)):
        _, v = _guarded(M * K, lead=lead)
        v.copy_(_dev(a.reshape(-1)))
        assert v.data_ptr() % 16 == 4
        ins[name] = v
    o = H.SpMMB200(g, K)
    o.preprocess(ins["vin"], torch.empty(M * K, device=DEV))
    t = o.transposed()
    for op in ("amax", "amin"):
        vb, vout = _guarded(M * K, lead=lead)
        ab, arg = _guarded(M * K, torch.int32, lead=lead)
        o.reduce(op, ins["vin"], vout, arg)
        dbb, db = _guarded(M * K, lead=lead)
        dvb, dval = _guarded(nnz, lead=lead)
        t.reduce_backward(ins["dc"], arg, db=db, dval=dval, vin=ins["vin"])
        torch.cuda.synchronize()
        for buf, n in ((vb, M * K), (ab, M * K), (dbb, M * K), (dvb, nnz)):
            assert _untouched(buf, lead, n), op
        want_v, want_a = RO.reduce_f32(ptr, idx, val, vin, K, op)
        an = arg.cpu().numpy().reshape(M, K)
        assert _same(vout.cpu().numpy().reshape(M, K), want_v) and np.array_equal(an, want_a), op
        want_db, want_dv = RO.reduce_backward_f32(ptr, idx, val, dcn, an, vin, M, K)
        assert _same(db.cpu().numpy().reshape(M, K), want_db) and _same(dval.cpu().numpy(), want_dv), op
        assert np.isnan(want_v).any() and np.isinf(want_v).any()
    t.close()
    o.close()
