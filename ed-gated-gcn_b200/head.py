"""The classifier head and its loss as modules the fused block recognises.

Reference: ``self.dense = nn.Linear(2 * hidden, polarities)`` applied to ``torch.cat([aspect, pooled], 1)``
(models/bert_amir5.py:573, :643) and ``criterion = nn.CrossEntropyLoss()`` (train.py:96, :121).  Both are
``[B, *]``-sized work that torch runs as a dozen small library launches between the forward and the backward pass of
the block; here the head runs on the block head's kernels with the fc part left out (``edg_block_head_fwd``, and
``edg_block_head_bwd`` + ``edg_block_head_wgrad`` backward) and the loss is two (``edg_cross_entropy_fwd/bwd``).
"""
from __future__ import annotations

import torch
import torch.nn as nn

from . import _lib as L
from . import ops


class _DenseHeadFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, a, p, weight, bias):
        ctx.save_for_backward(a, p, weight)
        ctx.has_bias = bias is not None
        return ops.block_head_fwd(a, None, p, None, weight, bias, None, None)[1]

    @staticmethod
    def backward(ctx, g):
        a, p, weight = ctx.saved_tensors
        da = dp = None
        if ctx.needs_input_grad[0] or ctx.needs_input_grad[1]:
            _, da, dp = ops.block_head_bwd(None, a, None, False, weight, None, None, g_logits=g)
        dW, db, _, _ = ops.block_head_wgrad(None, g, a, None, p, want_bias=ctx.has_bias)
        return (da.to(a.dtype) if da is not None else None, dp.to(p.dtype) if dp is not None else None,
                dW.to(weight.dtype), db)


class DenseHead(nn.Linear):
    """``nn.Linear(2 * hidden, n_classes)`` called as ``head(aspect [B,D], pooled [B,D]) -> logits [B,C]``: the
    reference's ``self.dense(torch.cat([aspect, pooled], 1))`` with the same parameter names and shapes (``weight
    [C, 2D]``, ``bias [C]``), so a reference checkpoint loads unchanged.  Passed as ``logits_fn`` to
    :class:`GatedGCNStack` it is recognised and run by the block's own kernels (no inner autograd graph, no
    ``head_params`` to declare); called on its own it is an autograd function over the same kernels."""

    def fusable(self, D: int) -> bool:
        return (self.in_features == 2 * D and self.out_features <= ops.DENSE_HEAD_MAX_CLASSES
                and self.weight.dtype == torch.float32 and self.weight.is_cuda)

    def forward(self, a: torch.Tensor, p: torch.Tensor = None) -> torch.Tensor:   # noqa: D401
        if p is None:                       # plain nn.Linear call on an already concatenated input
            return super().forward(a)
        if not a.is_cuda:
            raise L.EdgError("libedgcn takes CUDA tensors only (there is no CPU path)")
        return _DenseHeadFn.apply(a, p, self.weight, self.bias)


class _CrossEntropyFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, logits, target, ignore_index):
        lg = logits.detach()
        lg = lg if (lg.dtype == torch.float32 and lg.stride(1) == 1) else lg.float().contiguous()
        tgt = target if (target.dtype == torch.int64 and target.is_contiguous()) else target.long().contiguous()
        out, bad = ops.cross_entropy_fwd(lg, tgt, ignore_index)
        ctx.save_for_backward(lg, tgt, out)
        ctx.ignore_index, ctx.in_dtype, ctx.bad = ignore_index, logits.dtype, bad
        return out[0]

    @staticmethod
    def backward(ctx, g):
        lg, tgt, out = ctx.saved_tensors
        gs = g if (g.dtype == torch.float32 and g.is_cuda) else g.float().to(lg.device)
        dlg = ops.cross_entropy_bwd(lg, tgt, gs.reshape(1), out, ctx.ignore_index)
        return dlg.to(ctx.in_dtype), None, None


def cross_entropy(logits: torch.Tensor, target: torch.Tensor, ignore_index: int = -100) -> torch.Tensor:
    """``nn.CrossEntropyLoss()(logits, target)`` (mean over the targets that are not ``ignore_index``) in two launches.
    Targets outside ``[0, C)`` are not counted and leave a zero gradient row (torch raises a device assert there)."""
    if not logits.is_cuda:
        raise L.EdgError("libedgcn takes CUDA tensors only (there is no CPU path)")
    assert logits.dim() == 2 and target.shape == (logits.shape[0],)
    return _CrossEntropyFn.apply(logits, target, int(ignore_index))


class CrossEntropyLoss(nn.Module):
    """Drop-in for the reference's ``criterion`` (train.py:96)."""

    def __init__(self, ignore_index: int = -100):
        super().__init__()
        self.ignore_index = ignore_index

    def forward(self, logits, target):
        return cross_entropy(logits, target, self.ignore_index)


class _TotalLossFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, ce, xy, kl, gate_w, kl_w):
        def dev_scalar(t):
            if not torch.is_tensor(t):
                return None                       # the ungated ablation returns xy = 0.0 (bert_amir5.py:742)
            t = t.detach()
            return t if t.dtype == torch.float32 else t.float()
        terms = [dev_scalar(ce), dev_scalar(xy), dev_scalar(kl)]
        out = torch.empty((1,), dtype=torch.float32, device=terms[0].device)
        L.call("edg_loss_combine", L.ptr(terms[0]), L.ptr(terms[1]), L.ptr(terms[2]), 1.0, float(gate_w), float(kl_w),
               L.ptr(out), L.stream())
        ctx.w = (1.0, float(gate_w), float(kl_w))
        ctx.is_t = [t is not None for t in terms]
        ctx.shapes = [tuple(t.shape) if t is not None else None for t in terms]
        return out[0]

    @staticmethod
    def backward(ctx, g):
        g = g if (g.dtype == torch.float32 and g.is_cuda) else g.float().cuda()
        o3 = torch.empty((3,), dtype=torch.float32, device=g.device)
        L.call("edg_loss_combine_bwd", L.ptr(g.reshape(1)), ctx.w[0], ctx.w[1], ctx.w[2], L.ptr(o3), L.stream())
        return tuple(o3[i].reshape(ctx.shapes[i]) if ctx.is_t[i] else None for i in range(3)) + (None, None)


def total_loss(ce: torch.Tensor, xy, kl, gate_weight: float, kl_weight: float) -> torch.Tensor:
    """``loss = ce + gate_weight * xy + kl_weight * kl`` (train.py:115-118) in one launch forward and one backward
    (torch: two multiplies + two adds, and as many again in the backward pass, each a launch on the critical path)."""
    if not ce.is_cuda:
        raise L.EdgError("libedgcn takes CUDA tensors only (there is no CPU path)")
    return _TotalLossFn.apply(ce, xy, kl, gate_weight, kl_weight)
