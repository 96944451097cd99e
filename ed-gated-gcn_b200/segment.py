"""Segment reductions next to the gated block on the same packed layout (SURVEY.md 8f).

* ``wordpiece_mean`` -- N1: the ``torch.bmm(transform, x)`` that averages word pieces into words
  (models/bert_amir5.py:600, bert_ed.py:50, bertdm.py:166; transform built at data_utils.py:438-451 with ``1/l``
  entries over the ``l`` contiguous pieces of a word) as a segment mean over contiguous rows;
  ``transform_bmm`` keeps the reference's dense ``[B,T,L] x [B,L,D]`` call shape.
* ``lr_pool`` -- N4: BertDM's left/right max-pooling around the trigger (models/bertdm.py:116-140, :174-185).
* ``span_max`` -- the trigger vector of BertAmir / BertAmir2: max-pool of the LSTM output over the trigger's word
  pieces (``torch.max(x.masked_fill(aspect_mask, -1e12), 1)``, models/bert_amir.py:118, :259) as a max over one
  contiguous run of rows per sentence.

CUDA tensors only; no fallback.
"""
from __future__ import annotations

from typing import Optional, Tuple

import torch

from . import _lib as L
from . import ops
from .gcn import _compute_dtype


class _SegmentMeanFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, seg_start, seg_len, cdtype):
        xr = ops.as_rows(x, cdtype)
        P, D = xr.shape
        N = seg_start.numel()
        y = ops.alloc_rows(N, D, cdtype, x.device, min_ld=ops.row_pitch(D, cdtype))
        L.call("edg_segment_mean", L.ptr(xr), L.dt(xr), ops.ld(xr), L.ptr(seg_start), L.ptr(seg_len), N, D, L.ptr(y),
               L.dt(y), ops.ld(y), L.stream())
        ctx.save_for_backward(seg_start, seg_len)
        ctx.meta = (P, D, cdtype, x.dtype)
        return y

    @staticmethod
    def backward(ctx, gy):
        seg_start, seg_len = ctx.saved_tensors
        P, D, cd, xdt = ctx.meta
        g = ops.as_rows(gy, cd)
        dx = ops.alloc_rows(P, D, cd, gy.device)
        L.call("edg_segment_mean_bwd", L.ptr(g), L.dt(g), ops.ld(g), L.ptr(seg_start), L.ptr(seg_len), seg_start.numel(), D,
               L.ptr(dx), ops.ld(dx), P, L.stream())
        return (dx if dx.dtype == xdt else dx.to(xdt)), None, None, None


def wordpiece_mean(x_pieces: torch.Tensor, seg_start: torch.Tensor, seg_len: torch.Tensor,
                   compute_dtype=None) -> torch.Tensor:
    """x_pieces ``[P,D]`` packed word-piece rows, word ``i`` = mean of rows ``seg_start[i] .. +seg_len[i]``
    -> ``[N,D]`` packed word rows (``y = transform @ x`` with the 1/l transform of data_utils.py:438-451)."""
    if not x_pieces.is_cuda:
        raise L.EdgError("wordpiece_mean runs on CUDA tensors only (there is no CPU path)")
    cd = _compute_dtype(compute_dtype) if compute_dtype is not None else (
        x_pieces.dtype if x_pieces.dtype in L.DTYPES else torch.float32)
    dev = x_pieces.device
    return _SegmentMeanFn.apply(x_pieces, seg_start.to(device=dev, dtype=torch.int32).contiguous(),
                                seg_len.to(device=dev, dtype=torch.int32).contiguous(), cd)


def segments_from_transform(transform: torch.Tensor, check: bool = True) -> Tuple[torch.Tensor, torch.Tensor]:
    """Dense ``[B,T,L]`` transform (inputs['transform'][:, :T, :L], bert_amir5.py:586) -> ``seg_start``,
    ``seg_len`` int32 ``[B*T]`` addressing the rows of ``x.reshape(B*L, D)``.  All-zero rows (padding words)
    become empty segments.  ``check`` verifies what data_utils.py:438-451 guarantees: each row is a contiguous
    run of equal entries ``1/len``."""
    B, T, Lb = transform.shape
    nz = transform != 0
    seg_len = nz.sum(2)
    first = torch.argmax(nz.to(torch.int8), dim=2)
    if check:
        last = Lb - 1 - torch.argmax(nz.flip(2).to(torch.int8), dim=2)
        contiguous = ((last - first + 1 == seg_len) | (seg_len == 0)).all()
        want = torch.where(seg_len > 0, 1.0 / seg_len.clamp(min=1).float(), torch.zeros((), device=transform.device))
        uniform = (torch.where(nz, transform.float(), want[..., None]) == want[..., None]).all()
        if not (bool(contiguous) and bool(uniform)):
            raise L.EdgError("transform is not a word-piece averaging matrix (contiguous runs of 1/len per row)")
    off = torch.arange(B, device=transform.device)[:, None] * Lb
    return (first + off).reshape(-1).to(torch.int32), seg_len.reshape(-1).to(torch.int32)


def transform_bmm(transform: torch.Tensor, x: torch.Tensor, compute_dtype=None, check: bool = True) -> torch.Tensor:
    """Drop-in for ``torch.bmm(transform, x)`` (bert_amir5.py:600): transform ``[B,T,L]``, x ``[B,L,D]`` ->
    ``[B,T,D]``; padding words (all-zero transform rows) give zero rows, as in the reference."""
    B, T, Lb = transform.shape
    if x.shape[0] != B or x.shape[1] != Lb:
        raise L.EdgError(f"transform {tuple(transform.shape)} does not match x {tuple(x.shape)}")
    s, n = segments_from_transform(transform, check=check)
    y = wordpiece_mean(x.reshape(B * Lb, x.shape[2]), s, n, compute_dtype)
    return y.reshape(B, T, x.shape[2])


class _LRPoolFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, h, sent_ptr, anchor, T_pad, cdtype):
        hr = ops.as_rows(h, cdtype)
        N, D = hr.shape
        B = anchor.numel()
        pooled = torch.empty((B, 2 * D), dtype=torch.float32, device=h.device)
        arg = torch.empty((B, 2 * D), dtype=torch.int32, device=h.device)
        L.call("edg_lr_pool_fwd", L.ptr(hr), L.dt(hr), ops.ld(hr), L.ptr(sent_ptr), L.ptr(anchor), B, D, int(T_pad),
               L.ptr(pooled), L.ptr(arg), L.stream())
        ctx.save_for_backward(arg)
        ctx.meta = (N, D, cdtype, h.dtype)
        ctx.mark_non_differentiable(arg)
        return pooled, arg

    @staticmethod
    def backward(ctx, g, _garg=None):
        (arg,) = ctx.saved_tensors
        N, D, cd, hdt = ctx.meta
        dh = ops.alloc_rows(N, D, cd, g.device, zero=True)
        L.call("edg_lr_pool_bwd", L.ptr(g.float().contiguous()), L.ptr(arg), arg.shape[0], D, L.ptr(dh), L.dt(dh),
               ops.ld(dh), L.stream())
        return (dh if dh.dtype == hdt else dh.to(hdt)), None, None, None, None


class _LRPoolPairsFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, h, sent_ptr, pair_ptr, anchor, T_pad, cdtype):
        hr = ops.as_rows(h, cdtype)
        N, D = hr.shape
        S, P = sent_ptr.numel() - 1, anchor.numel()
        pooled = torch.empty((P, 2 * D), dtype=torch.float32, device=h.device)
        arg = torch.empty((P, 2 * D), dtype=torch.int32, device=h.device)
        L.call("edg_lr_pool_pairs_fwd", L.ptr(hr), L.dt(hr), ops.ld(hr), L.ptr(sent_ptr), L.ptr(pair_ptr), L.ptr(anchor), S,
               P, D, int(T_pad), L.ptr(pooled), L.ptr(arg), L.stream())
        ctx.save_for_backward(arg, sent_ptr, pair_ptr)
        ctx.meta = (N, D, cdtype, h.dtype)
        ctx.mark_non_differentiable(arg)
        return pooled, arg

    @staticmethod
    def backward(ctx, g, _garg=None):
        arg, sent_ptr, pair_ptr = ctx.saved_tensors
        N, D, cd, hdt = ctx.meta
        dh = ops.alloc_rows(N, D, cd, g.device)            # every sentence row is written by the kernel
        L.call("edg_lr_pool_pairs_bwd", L.ptr(g.float().contiguous()), L.ptr(arg), L.ptr(sent_ptr), L.ptr(pair_ptr),
               sent_ptr.numel() - 1, arg.shape[0], D, L.ptr(dh), L.dt(dh), ops.ld(dh), L.stream())
        return (dh if dh.dtype == hdt else dh.to(hdt)), None, None, None, None, None


def lr_pool(h: torch.Tensor, graph, anchor_index: torch.Tensor, T_pad: Optional[int] = None, compute_dtype=None,
            return_arg: bool = False, pairs=None):
    """BertDM dynamic pooling (bertdm.py:174-185) on packed rows: ``[B, 2D]`` = ``cat(pooledL, pooledR) - 1``.
    ``T_pad`` = the padded length the reference would use (``sentence_length.max()``, bertdm.py:148; default
    ``graph.max_len``): it decides whether the left pool sees a masked zero.

    With ``pairs`` (a :class:`TriggerPairs` over ``graph``), ``h`` holds every sentence once (``graph.n_rows`` rows),
    ``anchor_index`` is the sentence-local anchor of every pair (``[P]``, usually ``pairs.anchor``) and the result is
    ``[P, 2D]`` in pair order: bit for bit what the call gives on the expanded batch (each sentence's rows copied once
    per pair), with ``arg`` naming sentence rows.  Each sentence's rows are read twice, not once per pair, and the
    gradient sums over a sentence's pairs in ascending pair order.  The default ``T_pad`` = ``graph.max_len`` is the
    expanded batch's padded length whenever every sentence has a pair, as in every
    ``collate_packed(group_sentences=True)`` batch; a caller with pair-less sentences passes the expanded batch's
    ``T_pad`` (its longest sentence that has a pair).  The trigger row of each pair stays a row gather:
    ``words[pairs.pair_start + pairs.anchor]``."""
    if not h.is_cuda:
        raise L.EdgError("lr_pool runs on CUDA tensors only (there is no CPU path)")
    cd = _compute_dtype(compute_dtype) if compute_dtype is not None else (h.dtype if h.dtype in L.DTYPES else torch.float32)
    anchor = anchor_index.to(device=h.device, dtype=torch.int32).contiguous()
    T_pad = T_pad if T_pad is not None else graph.max_len
    if pairs is None:
        pooled, arg = _LRPoolFn.apply(h, graph.sent_ptr, anchor, T_pad, cd)
    else:
        if pairs.n_sentences != graph.n_graphs:
            raise L.EdgError(f"pairs cover {pairs.n_sentences} sentences, the graph has {graph.n_graphs}")
        if h.dim() != 2 or h.shape[0] != graph.n_rows:
            raise L.EdgError(f"with pairs, h must hold every sentence once: [{graph.n_rows}, D], got {tuple(h.shape)}")
        if anchor.dim() != 1 or anchor.numel() != pairs.n_pairs:
            raise L.EdgError(f"anchor_index must give one anchor per pair: [{pairs.n_pairs}], got {tuple(anchor.shape)}")
        pooled, arg = _LRPoolPairsFn.apply(h, graph.sent_ptr, pairs.pair_ptr, anchor, T_pad, cd)
    return (pooled, arg) if return_arg else pooled


class _SpanMaxFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, span_start, span_len, max_len, cdtype):
        from .graph import DepGraph
        xr = ops.as_rows(x, cdtype)
        P, D = xr.shape
        B = span_start.numel()
        dev = x.device
        # the pooling kernel works on a partition of the rows into "sentences": gap, span, gap, span, ..., gap
        sp = torch.empty(2 * B + 2, dtype=torch.int32, device=dev)
        sp[0] = 0
        sp[1:-1:2] = span_start
        sp[2:-1:2] = span_start + span_len
        sp[-1] = P
        row_sent = torch.bucketize(torch.arange(P, device=dev, dtype=torch.int32), sp[1:].contiguous(), right=True).int()
        g = DepGraph(sp, sp, sp, row_sent, 2 * B + 1, P, int(max_len))           # (row_ptr / col are not used by pooling)
        ones = torch.ones((1, 2 * B + 1, D), dtype=torch.float32, device=dev)
        pooled, arg = ops.pool_fwd(xr, g, ones)
        pooled, arg = pooled[0, 1::2].contiguous(), arg[0, 1::2].contiguous()
        empty = (span_len == 0)[:, None]
        pooled = torch.where(empty, torch.full_like(pooled, -1e12), pooled)      # an all-masked row pools to the fill value
        ctx.save_for_backward(torch.where(empty, torch.full_like(arg, -1), arg))
        ctx.meta = (P, D, cdtype, x.dtype)
        return pooled

    @staticmethod
    def backward(ctx, g):
        (arg,) = ctx.saved_tensors
        P, D, cd, xdt = ctx.meta
        dx = ops.alloc_rows(P, D, torch.float32, g.device, zero=True)
        ld = dx.stride(0)
        flat = dx.as_strided((P * ld,), (1,))
        ok = arg >= 0
        idx = (arg.long().clamp_min(0) * ld + torch.arange(D, device=g.device)[None, :])[ok]
        flat.index_add_(0, idx, g.float()[ok])                                   # one target per (sentence, column): no duplicates
        return (dx if dx.dtype == xdt else dx.to(xdt)), None, None, None, None


def span_max(x_rows: torch.Tensor, span_start: torch.Tensor, span_len: torch.Tensor, max_len: Optional[int] = None,
             compute_dtype=None) -> torch.Tensor:
    """``[B,D]`` = max over rows ``span_start[b] .. +span_len[b]`` of the packed rows ``x_rows [P,D]`` (first row wins
    ties, as ``torch.max``); spans ascending and disjoint (one per sentence).  For ``x [B,L,D]`` with the reference's
    ``aspect_mask`` (zeros on the trigger's word pieces, data_utils.py:470-472): ``span_start = b*L + first zero``,
    ``span_len = number of zeros``.  ``max_len`` = longest run between span boundaries (sizes the staging window; read
    back from the device when omitted)."""
    if not x_rows.is_cuda:
        raise L.EdgError("span_max runs on CUDA tensors only (there is no CPU path)")
    cd = _compute_dtype(compute_dtype) if compute_dtype is not None else (x_rows.dtype if x_rows.dtype in L.DTYPES else torch.float32)
    dev = x_rows.device
    s = span_start.to(device=dev, dtype=torch.int32).contiguous()
    n = span_len.to(device=dev, dtype=torch.int32).contiguous()
    if max_len is None:
        bounds = torch.cat([torch.zeros(1, dtype=torch.int32, device=dev), torch.stack([s, s + n], 1).reshape(-1),
                            torch.full((1,), x_rows.shape[0], dtype=torch.int32, device=dev)])
        max_len = int((bounds[1:] - bounds[:-1]).max().item())
    return _SpanMaxFn.apply(x_rows, s, n, max_len, cd)
