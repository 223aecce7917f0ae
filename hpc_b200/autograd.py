"""Differentiable SpMM and graph attention as torch.autograd operations over the engine's kernels.

GraphSpMM: forward is `run`; backward gives dB = Aᵀ·dC through the transposed operator and dval (the gradient for A's
edge values) through `sddmm(dC, B)`, each only when it is needed.

GraphAttention: scores = sddmm(q, k), alpha = edge_softmax(scores), out = A_alpha·v, with A_alpha the graph's pattern
carrying alpha as edge values; every step differentiable.
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


class GraphSpMM:
    """C = A·B for the CSR `g` (num_v x b_rows) and a dense B (b_rows x feat_in), differentiable in B and in g.val.

    options are passed to the forward operator (SpMMB200), e.g. b_rows for a row block. g.val may require grad
    (learned edge weights); an in-place change of g.val (an optimizer step) is noticed through its version counter and
    re-staged into the operators before the next forward. Call close() when done (or rely on garbage collection)."""

    def __init__(self, g: CSR, feat_in: int, **options):
        self.g = g
        self.feat_in = int(feat_in)
        self.op = SpMMB200(g, self.feat_in, **options)
        self._t = None
        self._staged = None
        self._prepared = False

    def transposed(self) -> SpMMB200:
        """The operator over Aᵀ (created and planned on first use)."""
        if self._t is None:
            self._t = self.op.transposed(self.feat_in)
            dc = torch.empty((self.op.num_v, self.feat_in), dtype=torch.float32, device=self.g.ptr.device)
            db = torch.empty((self.op.b_rows, self.feat_in), dtype=torch.float32, device=self.g.ptr.device)
            self._t.preprocess(dc, db)
        return self._t

    def _stage(self, b: torch.Tensor) -> None:
        version = self.g.val._version
        if not self._prepared:
            c = torch.empty((self.g.num_v, self.feat_in), dtype=torch.float32, device=b.device)
            self.op.preprocess(b, c)
            self._prepared = True
        elif version != self._staged:
            self.op.refresh_values()
            if self._t is not None:
                self._t.refresh_values()
        self._staged = version

    def __call__(self, b: torch.Tensor) -> torch.Tensor:
        if b.dtype != torch.float32 or not b.is_cuda or b.shape != (self.op.b_rows, self.feat_in):
            raise ValueError(f"B: need a CUDA float32 tensor of shape ({self.op.b_rows}, {self.feat_in})")
        b = b.contiguous()
        self._stage(b)
        return _GraphSpMMFn.apply(self, b, self.g.val)

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


def _stage(mod, values, op):
    """Puts `values` into the attention module's edge-value buffer and re-stages `op`'s panels from it. Done before every
    run: autograd interleaves the backwards of several calls, so nothing can be assumed about what is staged."""
    mod._val.copy_(values)
    op.refresh_values()


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
            _stage(mod, ds, mod.op)
            mod.op.run(k, dq)
        if ctx.needs_input_grad[2]:   # dk = S_dsᵀ·q
            dk = torch.empty_like(k)
            t = mod.transposed()
            _stage(mod, ds, t)
            t.run(q, dk)
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
        op = mod._op()
        _stage(mod, alpha, op)
        op.run(v, out)
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
            t = mod.transposed()
            _stage(mod, alpha, t)
            t.run(dout, dv)
        return None, dalpha, dv


class GraphAttention:
    """Dot-product attention over the CSR pattern of `g` (num_v x b_rows): out = softmax_row(<q_r, k_c>)·v, with
    q: num_v x feat_in, k and v: b_rows x feat_in (CUDA float32). Differentiable in q, k and v, and through the separate
    steps scores / softmax / aggregate (e.g. GAT scores built in torch, then softmax and aggregate). The caller scales q.

    Uses g.ptr / g.idx only: the edge values of every run are the module's own buffer, so g.val is never read or
    written. options are passed to the forward operator (SpMMB200), e.g. b_rows for a row block. The forward operator
    is planned on first use, the transposed one is created when a gradient first needs it. Call close() when done (or
    rely on garbage collection)."""

    def __init__(self, g: CSR, feat_in: int, **options):
        self.g = g
        self.feat_in = int(feat_in)
        self._val = torch.zeros(g.num_e, dtype=torch.float32, device=g.ptr.device)
        self.op = SpMMB200(CSR(g.num_v, g.num_e, g.ptr, g.idx, self._val), self.feat_in, **options)
        self._t = None
        self._prepared = False

    def _op(self) -> SpMMB200:
        """The forward operator, planned on first use."""
        if not self._prepared:
            dev = self.g.ptr.device
            b = torch.empty((self.op.b_rows, self.feat_in), dtype=torch.float32, device=dev)
            c = torch.empty((self.g.num_v, self.feat_in), dtype=torch.float32, device=dev)
            self.op.preprocess(b, c)
            self._prepared = True
        return self.op

    def transposed(self) -> SpMMB200:
        """The operator over the pattern's transpose (created and planned on first use); it reads the module's edge-value
        buffer through refresh_values."""
        if self._t is None:
            op = self._op()
            self._t = op.transposed(self.feat_in)
            dev = self.g.ptr.device
            dc = torch.empty((op.num_v, self.feat_in), dtype=torch.float32, device=dev)
            db = torch.empty((op.b_rows, self.feat_in), dtype=torch.float32, device=dev)
            self._t.preprocess(dc, db)
        return self._t

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
