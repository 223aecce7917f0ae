"""How operators are made, checked and planned, on the GPU.

- GraphSpMM and GraphAttention plan their operators without torch allocations: preprocess's vin / vout are hints the
  library never reads, and plans live in the library's own pool.
- Every SpMMB200 method refuses a tensor on the wrong device, of the wrong dtype, non-contiguous or too short with a
  ValueError that names the argument, before anything reaches the library.
- A transposed operator that cannot be built (a column outside B) leaves the device usable for the next one.
"""
import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

if not torch.cuda.is_available():
    pytest.skip("no CUDA device", allow_module_level=True)

import hpc_b200 as H  # noqa: E402
from oracle import cpu as O  # noqa: E402

DEV = "cuda"


def _csr(ptr, idx):
    return H.CSR(len(ptr) - 1, len(idx), torch.from_numpy(np.ascontiguousarray(ptr, np.int32)).to(DEV),
                 torch.from_numpy(np.ascontiguousarray(idx, np.int32)).to(DEV),
                 H.fill_normal(torch.empty(max(len(idx), 1), device=DEV), 123, 1))


def _dense(rows, K, stream):
    return H.fill_normal(torch.empty(rows * K, device=DEV), 123, stream).reshape(rows, K)


def test_planning_allocates_no_tensors():
    """Planning through the modules' lazy entry points, before any call, leaves torch's peak allocation where it was.
    The first call then still stages the values g.val holds at that call (forward and transposed)."""
    M, deg, K = 1 << 17, 8, 128   # b_rows x K floats: 64 MiB
    rng = np.random.default_rng(7)
    g = _csr(np.arange(M + 1, dtype=np.int64) * deg, rng.integers(0, M, M * deg))
    mods = [H.GraphAttention(g, K), H.GraphSpMM(g, K), H.GraphSpMM(g, K, reduce="amax")]
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    before = torch.cuda.max_memory_allocated()
    for m in mods:
        m._op()
        m.transposed()
        torch.cuda.synchronize()
        assert torch.cuda.max_memory_allocated() == before, type(m).__name__
    for m in mods:
        m.op.plan_info()                    # planned (plan_select refuses a handle without a plan)
    mods[0].transposed().plan_info()
    mods[1].transposed().plan_info()
    with pytest.raises(H.SpmmB200Error):   # reduce_backward needs no plan: amax's transposed operator has none
        mods[2].transposed().plan_info()

    g.val.mul_(-0.5)                        # in place, after planning: the first call must read these values
    b = _dense(M, K, 2).requires_grad_(True)
    got = mods[1](b)
    got.sum().backward()
    fresh = H.GraphSpMM(g, K)
    b2 = b.detach().clone().requires_grad_(True)
    want = fresh(b2)
    want.sum().backward()
    assert torch.equal(got.detach().view(torch.int32), want.detach().view(torch.int32))
    assert torch.equal(b.grad.view(torch.int32), b2.grad.view(torch.int32))
    for m in mods + [fresh]:
        m.close()


def _bad_variants(t):
    """(what, tensor): t on the other device, of another dtype, non-contiguous, and one element short."""
    other = torch.device("cpu") if t.is_cuda else torch.device(DEV)
    wrong = torch.int64 if t.dtype == torch.int32 else torch.float64
    strided = torch.zeros(2 * t.numel(), dtype=t.dtype, device=t.device)[::2]
    return [("device", t.to(other)), ("dtype", t.to(wrong)), ("non-contiguous", strided),
            ("short", t.flatten()[: t.numel() - 1])]


def _refuses_each(call, args):
    """call(**args) with each argument in turn replaced by each bad variant raises ValueError naming it."""
    for name, t in args.items():
        for what, bad in _bad_variants(t):
            with pytest.raises(ValueError) as e:
                call(**{**args, name: bad})
            assert str(e.value).split(":")[0] in (name, "CSR." + name), (name, what, str(e.value))


def test_every_method_checks_its_tensors():
    ptr, idx = H.gen_named_graph("c0")
    M, nnz, K = len(ptr) - 1, len(idx), 8
    g = _csr(ptr, idx)
    op = H.SpMMB200(g, K, live_values=1)
    t = op.transposed()
    f = lambda n: torch.zeros(n, device=DEV)
    i = lambda n: torch.zeros(n, dtype=torch.int32, device=DEV)
    h = lambda n: torch.zeros(n)
    _refuses_each(lambda ptr, idx, val: H.CSR(M, nnz, ptr, idx, val), {"ptr": g.ptr, "idx": g.idx, "val": g.val})
    _refuses_each(op.preprocess, {"vin": f(M * K), "vout": f(M * K)})
    _refuses_each(op.run, {"vin": f(M * K), "vout": f(M * K)})
    _refuses_each(op.run_profiled, {"vin": f(M * K), "vout": f(M * K)})
    _refuses_each(op.run_values, {"val": f(nnz), "vin": f(M * K), "vout": f(M * K)})
    _refuses_each(op.sddmm, {"x_row": f(M * K), "x_col": f(M * K), "out": f(nnz)})
    _refuses_each(op.edge_softmax, {"scores": f(nnz), "out": f(nnz)})
    _refuses_each(op.edge_softmax_backward, {"p": f(nnz), "dp": f(nnz), "ds": f(nnz)})
    _refuses_each(lambda **a: op.reduce("amax", **a), {"vin": f(M * K), "vout": f(M * K), "arg": i(M * K)})
    _refuses_each(t.reduce_backward, {"dc": f(M * K), "arg": i(M * K), "db": f(M * K), "dval": f(nnz), "vin": f(M * K)})
    _refuses_each(op.run_host, {"h_vin": h(M * K), "h_vout": h(M * K)})
    _refuses_each(op.run_host_sharded, {"h_vin": h(M * K), "h_vout": h(M * K)})
    t.close()
    op.close()


def test_failed_transposed_leaves_the_device_usable():
    ptr, idx = H.gen_named_graph("c0")
    M, K = len(ptr) - 1, 32
    bad_idx = idx.copy()
    bad_idx[len(idx) // 2] = M                      # a column outside B
    bad = H.SpMMB200(_csr(ptr, bad_idx), K)
    with pytest.raises(H.SpmmB200Error) as e:
        bad.transposed()
    assert e.value.code == -1 and "column outside" in str(e.value)
    bad.close()
    H.trim_memory()

    g = _csr(ptr, idx)
    op = H.SpMMB200(g, K)
    t = op.transposed()
    dc, db = _dense(M, K, 3), torch.full((M, K), float("nan"), device=DEV)
    t.preprocess(dc, db)
    t.run(dc, db)
    torch.cuda.synchronize()
    got = db.cpu().numpy()
    want, ab = O.spmm_t_f32(ptr, idx, g.val.cpu().numpy(), dc.cpu().numpy(), K, with_abs=True)
    whole = np.setdiff1d(np.arange(M), sorted(t.heavy_row_set()))
    assert np.array_equal(got[whole].view(np.int32), want[whole].view(np.int32))
    assert np.all(np.abs(got.astype(np.float64) - want) <= 1e-5 * ab + 1e-30)
    t.close()
    op.close()
