"""Host-side mirror of the reference's SpMM operator interface.

  struct CSR            PA4/handout/include/util.h:120-129   -> class CSR
  class SpMM            PA4/handout/include/spmm_base.h:8-46 -> class SpMM
  class SpMMOpt         PA4/handout/include/spmm_opt.h:5-26  -> class SpMMB200 (the slot it fills)
  allocate<float>       PA4/handout/include/data.h:24-37     -> allocate / fill_normal
  valid(float*,float*)  PA4/handout/src/valid.cu:41-56       -> valid

Same names, argument meaning and call protocol (preprocess once, then run any number of
times; run is asynchronous on the current stream and the caller synchronises). All tensors
are CUDA tensors; only their data pointers cross the C ABI.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import numpy as np
import torch

from ._lib import PlanInfo, check, lib


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None and t.numel() > 0 else C.c_void_p(0)


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _check_tensor(name, t, n, dtype=torch.float32, cuda=True):
    """Raises ValueError naming `name` unless t is a contiguous tensor of `dtype` with >= n elements, on a CUDA device
    (cuda=True) or on the host (cuda=False)."""
    if t.is_cuda != cuda or t.dtype != dtype or not t.is_contiguous() or t.numel() < n:
        kind, dt = "CUDA" if cuda else "host", str(dtype).removeprefix("torch.")
        raise ValueError(f"{name}: need a contiguous {kind} {dt} tensor of >= {n} elements")


@dataclass
class CSR:
    """struct CSR: device pointers, int32 indices (util.h:120-129)."""

    num_v: int
    num_e: int
    ptr: torch.Tensor  # int32[num_v + 1]
    idx: torch.Tensor  # int32[num_e]
    val: torch.Tensor  # float32[num_e]

    def __post_init__(self):
        _check_tensor("CSR.ptr", self.ptr, self.num_v + 1, torch.int32)
        _check_tensor("CSR.idx", self.idx, self.num_e, torch.int32)
        _check_tensor("CSR.val", self.val, self.num_e)


class SpMM:
    """class SpMM (spmm_base.h:8-46): abstract operator over a borrowed CSR."""

    def __init__(self, g: CSR, feat_in: int):
        self.g = g
        self.num_v, self.num_e, self.feat_in = g.num_v, g.num_e, int(feat_in)

    def set_feat(self, feat_in: int) -> None:
        self.feat_in = int(feat_in)

    def preprocess(self, vin, vout) -> None:
        raise NotImplementedError

    def run(self, vin, vout) -> None:
        raise NotImplementedError


class SpMMB200(SpMM):
    """The engine, in the slot of SpMMOpt (PA4/handout/src/spmm_opt.cu:3-11)."""

    def __init__(self, g: CSR, feat_in: int, b_rows: int = 0, **options):
        """b_rows: rows of B when g is a row block of a larger graph (columns index the full B)."""
        super().__init__(g, feat_in)
        self.b_rows = int(b_rows) or g.num_v
        h = C.c_void_p()
        check(lib.spmm_b200_create(_ptr(g.ptr), _ptr(g.idx), _ptr(g.val), g.num_v, g.num_e,
                                   self.feat_in, C.byref(h)))
        self._h = h
        if self.b_rows != g.num_v:
            self.set_option("b_rows", self.b_rows)
        for k, v in options.items():
            self.set_option(k, v)

    def set_option(self, name: str, value: int) -> None:
        check(lib.spmm_b200_set_option(self._h, name.encode(), int(value)))

    def set_feat(self, feat_in: int) -> None:
        super().set_feat(feat_in)
        check(lib.spmm_b200_set_feat(self._h, self.feat_in))

    def _check_io(self, vin, vout, prefix="", cuda=True):
        _check_tensor(prefix + "vin", vin, self.b_rows * self.feat_in, cuda=cuda)
        _check_tensor(prefix + "vout", vout, self.num_v * self.feat_in, cuda=cuda)

    def _check_edges(self, **arrays):
        for name, t in arrays.items():
            _check_tensor(name, t, self.num_e)

    def set_gather(self, targets, row_offset: int, multicast: int = 0) -> None:
        """Stacked-layer epilogue: finished C rows also go to `targets` (device pointers as ints, or CUDA
        tensors) at row `row_offset`, or once through the NVLS `multicast` address. [] switches it off."""
        ptrs = [t.data_ptr() if hasattr(t, "data_ptr") else int(t) for t in targets]
        arr = (C.c_void_p * max(1, len(ptrs)))(*ptrs)
        check(lib.spmm_b200_set_gather(self._h, len(ptrs), arr, C.c_void_p(multicast or 0), int(row_offset)))

    def preprocess(self, vin, vout) -> None:
        self._check_io(vin, vout)
        self._plan()

    def _plan(self) -> None:
        """preprocess without vin / vout: the library takes them as hints only and reads neither."""
        check(lib.spmm_b200_preprocess(self._h, None, None, _stream()))

    def _derived(self, create, num_v: int, b_rows: int, feat_in: int | None, options: dict) -> "SpMMB200":
        """The operator that the C constructor `create` builds from this one's handle, with the given shape."""
        t = object.__new__(SpMMB200)
        t.g = None
        t.num_v, t.num_e, t.b_rows = num_v, self.num_e, b_rows
        t.feat_in = self.feat_in if feat_in is None else int(feat_in)
        h = C.c_void_p()
        check(create(self._h, t.feat_in, _stream(), C.byref(h)))
        t._h = h
        t._parent = self   # keeps the source operator (and the arrays it borrows) alive
        for k, v in options.items():
            t.set_option(k, v)
        return t

    def transposed(self, feat_in: int | None = None, **options) -> "SpMMB200":
        """The operator over A^T (spmm_b200_create_transposed): run(dC[num_v x K], dB[b_rows x K]) computes the gradient
        of this operator with respect to its input. The new operator owns its CSR; close it before this one."""
        return self._derived(lib.spmm_b200_create_transposed, self.b_rows, self.num_v, feat_in, options)

    def column_sorted(self, feat_in: int | None = None, **options) -> "SpMMB200":
        """The operator over the same matrix with every row in ascending column order (spmm_b200_create_column_sorted): for
        CSR inputs whose rows are not column-sorted, which otherwise stay in one column block. Results associate in column
        order. The new operator borrows ptr, owns idx / val; close it before this one."""
        return self._derived(lib.spmm_b200_create_column_sorted, self.num_v, self.b_rows, feat_in, options)

    def refresh_values(self) -> None:
        """Re-stage the plan's copy of idx/val after the caller changed them in place (same ptr)."""
        check(lib.spmm_b200_refresh_values(self._h, _stream()))

    def run(self, vin, vout) -> None:
        self._check_io(vin, vout)
        check(lib.spmm_b200_run(self._h, _ptr(vin), _ptr(vout), _stream()))

    def run_values(self, val, vin, vout) -> None:
        """run with the edge values `val` (spmm_b200_run_values): C = A_val·B, val[p] the value of the nonzero at CSR
        position p — on an operator from transposed() / column_sorted(), a position of the source operator, whose num_e
        values val holds. Needs the option live_values=1. Asynchronous on the current stream."""
        self._check_io(vin, vout)
        _check_tensor("val", val, self.num_e)
        check(lib.spmm_b200_run_values(self._h, _ptr(val), _ptr(vin), _ptr(vout), _stream()))

    def sddmm(self, x_row, x_col, out) -> None:
        """SDDMM over this operator's pattern (spmm_b200_sddmm): out[e] = <x_row[row(e)], x_col[idx[e]]> for every
        nonzero e, in CSR position order. x_row: num_v x feat_in, x_col: b_rows x feat_in, out: >= num_e floats.
        With x_row = dC and x_col = B, out is dL/dval of C = A·B. Asynchronous on the current stream."""
        _check_tensor("x_row", x_row, self.num_v * self.feat_in)
        _check_tensor("x_col", x_col, self.b_rows * self.feat_in)
        _check_tensor("out", out, self.num_e)
        check(lib.spmm_b200_sddmm(self._h, _ptr(x_row), _ptr(x_col), _ptr(out), _stream()))

    def edge_softmax(self, scores, out) -> None:
        """Softmax over each row's nonzeros (spmm_b200_edge_softmax), in CSR position order: out[e] = exp(s[e] - m_r) /
        sum_r exp(s - m_r). A row of -inf scores gives zeros. Needs no preprocess; out must not overlap scores.
        Asynchronous on the current stream."""
        self._check_edges(scores=scores, out=out)
        check(lib.spmm_b200_edge_softmax(self._h, _ptr(scores), _ptr(out), _stream()))

    def edge_softmax_backward(self, p, dp, ds) -> None:
        """The gradient of edge_softmax (spmm_b200_edge_softmax_backward): ds[e] = p[e] * (dp[e] - sum_r p * dp), with p
        its output. ds must not overlap p or dp. Asynchronous on the current stream."""
        self._check_edges(p=p, dp=dp, ds=ds)
        check(lib.spmm_b200_edge_softmax_backward(self._h, _ptr(p), _ptr(dp), _ptr(ds), _stream()))

    REDUCE_OPS = {"amax": 1, "amin": 2}   # SPMM_B200_REDUCE_AMAX / _AMIN

    def reduce(self, op: str, vin, vout, arg=None) -> None:
        """amax / amin aggregation over this operator's rows (spmm_b200_reduce): vout[r, j] = the winning message
        val[e] * vin[idx[e], j] over the nonzeros e of row r, arg[r, j] = e (int32, optional). NaN wins; ties go to the
        smaller CSR position; an empty row gives 0 and arg -1. vin: b_rows x feat_in, vout / arg: num_v x feat_in.
        Reads the current g.val (no refresh_values needed). Asynchronous on the current stream."""
        if op not in self.REDUCE_OPS:
            raise ValueError(f"reduce: op must be one of {sorted(self.REDUCE_OPS)}, got {op!r}")
        self._check_io(vin, vout)
        if arg is not None:
            _check_tensor("arg", arg, self.num_v * self.feat_in, torch.int32)
        check(lib.spmm_b200_reduce(self._h, self.REDUCE_OPS[op], _ptr(vin), _ptr(vout), _ptr(arg), _stream()))

    def reduce_backward(self, dc, arg, db=None, dval=None, vin=None) -> None:
        """The gradient of the source operator's reduce, on this operator, which must come from transposed()
        (spmm_b200_reduce_backward): db (the source's b_rows x feat_in) and dval (num_e, in the source's CSR positions),
        each optional, from dC and the forward's arg (both the source's num_v x feat_in). vin (the forward's B) is
        needed only with dval. Asynchronous on the current stream."""
        src_rows = self.b_rows   # this operator is Aᵀ: its b_rows are the source's rows
        _check_tensor("dc", dc, src_rows * self.feat_in)
        _check_tensor("arg", arg, src_rows * self.feat_in, torch.int32)
        if db is not None:
            _check_tensor("db", db, self.num_v * self.feat_in)
        if dval is not None:
            _check_tensor("dval", dval, self.num_e)
            if vin is None:
                raise ValueError("reduce_backward: dval needs vin (the forward's B)")
            _check_tensor("vin", vin, self.num_v * self.feat_in)
        check(lib.spmm_b200_reduce_backward(self._h, _ptr(dc), _ptr(arg), _ptr(vin), _ptr(db), _ptr(dval), _stream()))

    def run_profiled(self, vin, vout) -> float:
        """run + the kernel's device time in ms (synchronises)."""
        self._check_io(vin, vout)
        ms = C.c_float(0)
        check(lib.spmm_b200_run_profiled(self._h, _ptr(vin), _ptr(vout), _stream(), C.byref(ms)))
        return ms.value

    def run_host(self, h_vin: torch.Tensor, h_vout: torch.Tensor) -> None:
        """H2D(vin) -> run -> D2H(vout) -> sync, host (ideally pinned) float32 tensors."""
        self._check_io(h_vin, h_vout, "h_", cuda=False)
        check(lib.spmm_b200_run_host(self._h, C.c_void_p(h_vin.data_ptr()), C.c_void_p(h_vout.data_ptr()),
                                     _stream()))

    def set_replicate(self, world: int, rank: int, peers_b, multicast_b: int, peers_flags) -> None:
        """Sharded host I/O (spmm_b200_set_replicate): every rank's copy of B and flag words as mapped in this
        process (device pointers as ints), the NVLS multicast address of the B copies or 0."""
        pb = (C.c_void_p * max(1, world))(*[int(p) for p in peers_b])
        pf = (C.c_void_p * max(1, world))(*[int(p) for p in peers_flags])
        check(lib.spmm_b200_set_replicate(self._h, int(world), int(rank), pb, C.c_void_p(multicast_b or 0), pf))

    def run_host_sharded(self, h_vin: torch.Tensor, h_vout: torch.Tensor) -> int:
        """Collective over the ranks: upload this rank's share of B (h_vin is the whole B on the host), replicate it
        over NVLink, run, deliver the local block of C into h_vout, synchronise (spmm_b200_run_host_sharded).
        Returns the host-to-device bytes this rank copied."""
        self._check_io(h_vin, h_vout, "h_", cuda=False)
        check(lib.spmm_b200_run_host_sharded(self._h, C.c_void_p(h_vin.data_ptr()), C.c_void_p(h_vout.data_ptr()), _stream()))
        return int(lib.spmm_b200_replicate_h2d_bytes(self._h))

    @property
    def launches_per_run(self) -> int:
        return lib.spmm_b200_launches_per_run(self._h)

    def plan_info(self, col_block: int = 0) -> dict:
        check(lib.spmm_b200_plan_select(self._h, col_block))
        info = PlanInfo()
        check(lib.spmm_b200_plan_info(self._h, C.byref(info)))
        return info.as_dict()

    def plan_arrays(self, col_block: int = 0) -> dict:
        """One column block's plan, copied to host numpy arrays (parity tests compare these with the oracle)."""
        info = self.plan_info(col_block)
        out = {}
        nb = info["n_col_blocks"]
        for which, name, n in ((0, "row_perm", info["n_light"]), (1, "heavy_rows", info["n_heavy"]),
                               (2, "heavy_seg0", info["n_heavy"] + 1 if info["n_heavy"] else 0),
                               (3, "seg_desc", info["n_seg"] * 4), (4, "panel", info["panel_len"] * 2),
                               (5, "light_desc", info["n_light"] * 4), (6, "seg_hrow", info["n_seg"]),
                               (7, "split", (nb + 1) * self.num_v if nb > 1 else 0),
                               (8, "ltask", info["n_ltask"] * 2), (9, "lpanel", info["lpanel_len"] * 2),
                               (10, "utask", info["n_utask"] * 2), (12, "group_row", info["n_row_groups"] + 1)):
            a = np.empty(n, dtype=np.int32)
            check(lib.spmm_b200_plan_copy(self._h, which, a.ctypes.data_as(C.c_void_p), a.nbytes))
            out[name] = a
        out["seg_desc"] = out["seg_desc"].reshape(-1, 4)
        out["panel"] = out["panel"].reshape(-1, 2)
        out["light_desc"] = out["light_desc"].reshape(-1, 4)
        out["ltask"] = out["ltask"].reshape(-1, 2)
        out["utask"] = out["utask"].reshape(-1, 2)
        out["lpanel"] = out["lpanel"].reshape(-1, 2)
        if nb > 1:
            out["split"] = out["split"].reshape(nb + 1, self.num_v)
        return out

    def heavy_row_set(self) -> set:
        """Rows that are split into segments in ANY column block (re-associated sums)."""
        rows = set()
        for b in range(self.plan_info(0)["n_col_blocks"]):
            rows.update(self.plan_arrays(b)["heavy_rows"].tolist())
        return rows

    def close(self) -> None:
        if getattr(self, "_h", None):
            lib.spmm_b200_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:   # interpreter shutdown: the library may already be gone
            pass


def trim_memory() -> None:
    """Hand the plan memory pooled on the current device that no live operator uses back to the driver
    (`spmm_b200_trim_memory`)."""
    check(lib.spmm_b200_trim_memory())


def fill_normal(t: torch.Tensor, seed: int, stream_id: int, mean: float = 0.0, stddev: float = 0.1) -> torch.Tensor:
    """Counter-based N(mean, stddev) fill (the engine's stand-in for curandGenerateNormal, data.h:31)."""
    _check_tensor("fill_normal: t", t, 0)
    check(lib.spmm_b200_fill_normal(_ptr(t), t.numel(), seed, stream_id, mean, stddev, _stream()))
    return t


_alloc_counter = [0]


def allocate(num: int, seed: int = 123, random: bool = True, device="cuda") -> torch.Tensor:
    """allocate<float>(num) (data.h:24-37): rounded up to 512 elements, N(0, 0.1)-filled.
    Successive calls draw from successive streams, as successive curand calls do."""
    t = torch.empty((num + 511) // 512 * 512, dtype=torch.float32, device=device)
    if random:
        fill_normal(t, seed, _alloc_counter[0])
        _alloc_counter[0] += 1
    return t


def valid(y: torch.Tensor, y2: torch.Tensor, num: int) -> int:
    """valid(y, y2, num) (valid.cu:41-56): count of |(y - y2) / y| > 1e-2."""
    out = C.c_longlong(0)
    check(lib.spmm_b200_valid(_ptr(y), _ptr(y2), num, C.byref(out), _stream()))
    return out.value


def plan_host(ptr: np.ndarray, feat: int, seg_len: int = 0, reorder: bool = True) -> dict:
    """The row part of the plan from a host ptr array (spmm_b200_plan_host); no GPU needed."""
    ptr = np.ascontiguousarray(ptr, dtype=np.int32)
    m = len(ptr) - 1
    nl, nh, ns, pl = C.c_int(0), C.c_int(0), C.c_int(0), C.c_longlong(0)
    args = (C.c_void_p(ptr.ctypes.data), m, int(feat), int(seg_len), int(bool(reorder)))
    check(lib.spmm_b200_plan_host(*args, None, C.byref(nl), None, C.byref(nh), None, None, C.byref(ns), C.byref(pl)))
    row_perm = np.empty(nl.value, np.int32)
    heavy_rows = np.empty(nh.value, np.int32)
    heavy_seg0 = np.empty(nh.value + 1 if nh.value else 0, np.int32)
    seg_desc = np.empty(ns.value * 4, np.int32)
    vp = lambda a: C.c_void_p(a.ctypes.data)
    check(lib.spmm_b200_plan_host(*args, vp(row_perm), C.byref(nl), vp(heavy_rows), C.byref(nh), vp(heavy_seg0),
                                  vp(seg_desc), C.byref(ns), C.byref(pl)))
    return {"row_perm": row_perm, "heavy_rows": heavy_rows, "heavy_seg0": heavy_seg0,
            "seg_desc": seg_desc.reshape(-1, 4), "panel_len": pl.value}


def pack_light_host(cost: np.ndarray, groups: int, steps: int):
    """The light-stream packing rule on the host (spmm_b200_pack_light_host). -> (dst, ltask[n,2], lpanel_len)"""
    cost = np.ascontiguousarray(cost, dtype=np.int32)
    n = len(cost)
    nt, pl = C.c_int(0), C.c_longlong(0)
    cp = C.c_void_p(cost.ctypes.data) if n else None
    check(lib.spmm_b200_pack_light_host(cp, n, groups, steps, None, None, C.byref(nt), C.byref(pl)))
    dst = np.empty(n, np.int32)
    ltask = np.empty(nt.value * 2, np.int32)
    check(lib.spmm_b200_pack_light_host(cp, n, groups, steps, C.c_void_p(dst.ctypes.data) if n else None,
                                        C.c_void_p(ltask.ctypes.data) if nt.value else None, C.byref(nt), C.byref(pl)))
    return dst, ltask.reshape(-1, 2), pl.value
