"""Differentiable SpMM and graph attention as torch.autograd operations over the engine's kernels.

GraphSpMM: forward is `run`; backward gives dB = Aᵀ·dC through the transposed operator and dval (the gradient for A's
edge values) through `sddmm(dC, B)`, each only when it is needed. With reduce="amax" / "amin" the forward is `reduce`,
which also records the winning nonzero of every output, and the backward is `reduce_backward` on the transposed
operator; reduce="mean" divides the sum by the row's nonzero count.

GraphAttention: scores = sddmm(q, k), alpha = edge_softmax(scores), out = A_alpha·v, with A_alpha the graph's pattern
carrying alpha as edge values (run_values on live-value operators); every step differentiable.
"""
from __future__ import annotations

import torch

from .spmm import CSR, SpMMB200


class _GraphSpMMFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, mod, b, val):
        # `val` is g.val itself: passing it makes autograd route dval to it
        c = torch.empty((mod.g.num_v, mod.feat_in), dtype=torch.float32, device=b.device)
        mod.op.run(b, c)
        ctx.mod = mod
        ctx.save_for_backward(b)
        return c

    @staticmethod
    def backward(ctx, dc):
        mod = ctx.mod
        (b,) = ctx.saved_tensors
        dc = dc.contiguous()
        db = dval = None
        if ctx.needs_input_grad[1]:
            db = torch.empty_like(b)
            mod.transposed().run(dc, db)
        if ctx.needs_input_grad[2]:
            g = mod.g
            dval = torch.zeros_like(g.val)   # entries beyond num_e (if any) have no nonzero: zero
            mod.op.sddmm(dc, b, dval)
        return None, db, dval


class _GraphSpMMReduceFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, mod, b, val):
        # `val` is g.val itself: passing it makes autograd route dval to it
        c = torch.empty((mod.g.num_v, mod.feat_in), dtype=torch.float32, device=b.device)
        arg = torch.empty((mod.g.num_v, mod.feat_in), dtype=torch.int32, device=b.device)
        mod.op.reduce(mod.reduce, b, c, arg)
        ctx.mod = mod
        ctx.save_for_backward(b, arg)
        return c

    @staticmethod
    def backward(ctx, dc):
        mod = ctx.mod
        b, arg = ctx.saved_tensors
        db = torch.empty_like(b) if ctx.needs_input_grad[1] else None
        dval = torch.zeros_like(mod.g.val) if ctx.needs_input_grad[2] else None   # entries beyond num_e: zero
        if db is not None or dval is not None:
            mod.transposed().reduce_backward(dc.contiguous(), arg, db=db, dval=dval, vin=b if dval is not None else None)
        return None, db, dval


REDUCTIONS = ("sum", "mean", "amax", "amin")


class _Operators:
    """What GraphSpMM and GraphAttention share: the forward operator over g, planned on first use, and the operator over
    Aᵀ, created on first use and planned when the module runs on it. Plans live in the library's pool; close() releases
    both operators."""

    def __init__(self, g: CSR, feat_in: int, shared: dict, **options):
        """shared: the options of both operators; options: those of the forward one alone."""
        self.g = g
        self.feat_in = int(feat_in)
        self.op = SpMMB200(g, self.feat_in, **shared, **options)
        self._shared = shared
        self._t = None
        self._planned = False

    def _runs(self) -> bool:
        """Whether the module runs its operators (run / run_values, which need a plan on the transposed one too)."""
        return True

    def _op(self) -> SpMMB200:
        """The forward operator, planned on first use."""
        if not self._planned:
            self.op._plan()
            self._planned = True
        return self.op

    def transposed(self) -> SpMMB200:
        """The operator over Aᵀ (created on first use; planned when the module runs on it). On a live-value module its
        run_values takes edge values in g's CSR positions."""
        if self._t is None:
            self._t = self.op.transposed(self.feat_in, **self._shared)
            if self._runs():
                self._t._plan()
        return self._t

    def close(self) -> None:
        """Releases the transposed operator, then the forward one."""
        if self._t is not None:
            self._t.close()
            self._t = None
        self.op.close()

    def __del__(self):
        try:
            self.close()
        except Exception:   # interpreter shutdown: the library may already be gone
            pass


class GraphSpMM(_Operators):
    """C = A·B for the CSR `g` (num_v x b_rows) and a dense B (b_rows x feat_in), differentiable in B and in g.val.

    reduce (torch.sparse.mm's names): "sum" (default), "mean" (the sum over the row's nonzero count; empty rows give 0),
    "amax" / "amin" (per column, the largest / smallest val[e] * B[idx[e]] of the row; NaN wins, ties go to the
    smaller CSR position, empty rows give 0; the gradient goes to the winning nonzero alone).

    options are passed to the forward operator (SpMMB200), e.g. b_rows for a row block. g.val may require grad
    (learned edge weights); an in-place change of g.val (an optimizer step) is noticed through its version counter and
    re-staged into the operators before the next forward ("amax" / "amin" read g.val as it is). Call close() when done
    (or rely on garbage collection)."""

    def __init__(self, g: CSR, feat_in: int, reduce: str = "sum", **options):
        if reduce not in REDUCTIONS:
            raise ValueError(f"reduce must be one of {REDUCTIONS}, got {reduce!r}")
        super().__init__(g, feat_in, {}, **options)
        self.reduce = reduce
        self._staged = None
        self._deg = None

    def _runs(self) -> bool:
        """run reads the plan's copy of the values; reduce / reduce_backward read g.val itself, and reduce_backward
        needs no plan."""
        return self.reduce in ("sum", "mean")

    def _stage(self) -> None:
        version = self.g.val._version
        if self._planned and version != self._staged and self._runs():
            self.op.refresh_values()
            if self._t is not None:
                self._t.refresh_values()
        self._op()
        self._staged = version

    def _degrees(self) -> torch.Tensor:
        """Nonzeros per row as a (num_v, 1) float32 column, empty rows counted as 1 (their sum is 0)."""
        if self._deg is None:
            ptr = self.g.ptr[: self.g.num_v + 1]
            self._deg = (ptr[1:] - ptr[:-1]).clamp(min=1).to(torch.float32).unsqueeze(1)
        return self._deg

    def __call__(self, b: torch.Tensor) -> torch.Tensor:
        if b.dtype != torch.float32 or not b.is_cuda or b.shape != (self.op.b_rows, self.feat_in):
            raise ValueError(f"B: need a CUDA float32 tensor of shape ({self.op.b_rows}, {self.feat_in})")
        b = b.contiguous()
        self._stage()
        if self.reduce in ("amax", "amin"):
            return _GraphSpMMReduceFn.apply(self, b, self.g.val)
        c = _GraphSpMMFn.apply(self, b, self.g.val)
        return c / self._degrees() if self.reduce == "mean" else c


class _ScoresFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, mod, q, k):
        s = torch.empty(mod.g.num_e, dtype=torch.float32, device=q.device)
        mod._op().sddmm(q, k, s)
        ctx.mod = mod
        ctx.save_for_backward(q, k)
        return s

    @staticmethod
    def backward(ctx, ds):
        mod = ctx.mod
        q, k = ctx.saved_tensors
        ds = ds.contiguous()
        dq = dk = None
        if ctx.needs_input_grad[1]:   # dq = S_ds·k
            dq = torch.empty_like(q)
            mod.op.run_values(ds, k, dq)
        if ctx.needs_input_grad[2]:   # dk = S_dsᵀ·q
            dk = torch.empty_like(k)
            mod.transposed().run_values(ds, q, dk)
        return None, dq, dk


class _SoftmaxFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, mod, s):
        p = torch.empty_like(s)
        mod.op.edge_softmax(s, p)
        ctx.mod = mod
        ctx.save_for_backward(p)
        return p

    @staticmethod
    def backward(ctx, dp):
        (p,) = ctx.saved_tensors
        ds = torch.empty_like(p)
        ctx.mod.op.edge_softmax_backward(p, dp.contiguous(), ds)
        return None, ds


class _AggregateFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, mod, alpha, v):
        out = torch.empty((mod.g.num_v, mod.feat_in), dtype=torch.float32, device=v.device)
        mod._op().run_values(alpha, v, out)
        ctx.mod = mod
        ctx.save_for_backward(alpha, v)
        return out

    @staticmethod
    def backward(ctx, dout):
        mod = ctx.mod
        alpha, v = ctx.saved_tensors
        dout = dout.contiguous()
        dalpha = dv = None
        if ctx.needs_input_grad[1]:   # dalpha = sddmm(dout, v)
            dalpha = torch.empty_like(alpha)
            mod.op.sddmm(dout, v, dalpha)
        if ctx.needs_input_grad[2]:   # dv = A_alphaᵀ·dout
            dv = torch.empty_like(v)
            mod.transposed().run_values(alpha, dout, dv)
        return None, dalpha, dv


class GraphAttention(_Operators):
    """Dot-product attention over the CSR pattern of `g` (num_v x b_rows): out = softmax_row(<q_r, k_c>)·v, with
    q: num_v x feat_in, k and v: b_rows x feat_in (CUDA float32). Differentiable in q, k and v, and through the separate
    steps scores / softmax / aggregate (e.g. GAT scores built in torch, then softmax and aggregate). The caller scales q.

    The operators are built over g with live values: every run takes its edge values (alpha, or the score gradient) as
    an argument and reads them in the kernel, so nothing is staged between runs and g.val is never written. The
    transposed operator reads the same arrays, in g's CSR positions. options are passed to the forward operator
    (SpMMB200), e.g. b_rows for a row block. The forward operator is planned on first use, the transposed one is created
    when a gradient first needs it. Call close() when done (or rely on garbage collection)."""

    def __init__(self, g: CSR, feat_in: int, **options):
        super().__init__(g, feat_in, {"live_values": 1}, **options)

    def _dense(self, name, t, rows):
        if not isinstance(t, torch.Tensor) or t.dtype != torch.float32 or not t.is_cuda or t.shape != (rows, self.feat_in):
            raise ValueError(f"{name}: need a CUDA float32 tensor of shape ({rows}, {self.feat_in})")
        return t.contiguous()

    def _edges(self, name, t):
        if not isinstance(t, torch.Tensor) or t.dtype != torch.float32 or not t.is_cuda or t.shape != (self.g.num_e,):
            raise ValueError(f"{name}: need a CUDA float32 tensor of shape ({self.g.num_e},)")
        return t.contiguous()

    def scores(self, q: torch.Tensor, k: torch.Tensor) -> torch.Tensor:
        """s[e] = <q[row(e)], k[idx[e]]> for every nonzero (sddmm), in CSR position order."""
        q = self._dense("q", q, self.g.num_v)
        k = self._dense("k", k, self.op.b_rows)
        return _ScoresFn.apply(self, q, k)

    def softmax(self, s: torch.Tensor) -> torch.Tensor:
        """alpha = softmax of s over each row's nonzeros (edge_softmax); a row of -inf scores gives zeros."""
        return _SoftmaxFn.apply(self, self._edges("s", s))

    def aggregate(self, alpha: torch.Tensor, v: torch.Tensor) -> torch.Tensor:
        """out = A_alpha·v: the pattern with alpha as edge values times v (run)."""
        alpha = self._edges("alpha", alpha)
        v = self._dense("v", v, self.op.b_rows)
        return _AggregateFn.apply(self, alpha, v)

    def __call__(self, q: torch.Tensor, k: torch.Tensor, v: torch.Tensor) -> torch.Tensor:
        return self.aggregate(self.softmax(self.scores(q, k)), v)
