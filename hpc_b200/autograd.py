"""Differentiable SpMM: C = A·B as a torch.autograd operation over the engine's kernels.

Forward is `run`; backward gives dB = Aᵀ·dC through the transposed operator and dval (the gradient for A's edge values)
through `sddmm(dC, B)`, each only when it is needed.
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
