"""Drop-in ``GraphConvolution`` (reference: models/gcn.py:9-45).

Same constructor and ``forward(text, adj)`` signature, same parameter names and
shapes (``weight [in,out]``, ``bias [out]``; state-dict keys ``gc1.weight`` ...),
same result: ``adj @ (text @ W) / (rowsum(adj) + 1) + b`` with no activation.
The dense adjacency is converted once per batch to a packed CSR (cached, so
``gc2`` reuses ``gc1``'s conversion) and the layer runs as
``aggregate -> GEMM`` on hand-written sm_100a kernels.  CUDA tensors only.
"""
from __future__ import annotations

import math
import weakref
from typing import Optional

import torch
import torch.nn as nn

from . import _lib as L
from . import ops
from .graph import DepGraph, graph_from_dense

_COMPUTE = {"f32": torch.float32, "fp32": torch.float32, "float32": torch.float32,
            "bf16": torch.bfloat16, "bfloat16": torch.bfloat16}


def _compute_dtype(x) -> torch.dtype:
    if isinstance(x, torch.dtype):
        return x
    return _COMPUTE[str(x)]


# adjacency -> CSR cache: the reference calls gc1(x, adj) and gc2(gcn1, adj) with the SAME tensor object
# (bert_amir5.py:589, :626, :639).  Entries are tied to that object's lifetime (weak reference, identity checked on
# every hit) and to its version counter, so neither a freed-and-reallocated block at the same address (train.py:108
# makes a fresh `.to(device)` batch per step) nor an in-place edit can ever return a stale graph.
_GRAPH_CACHE: "dict[int, tuple]" = {}


def cached_graph_from_dense(adj: torch.Tensor) -> DepGraph:
    key = id(adj)
    ent = _GRAPH_CACHE.get(key)
    if ent is not None and ent[0]() is adj and ent[1] == adj._version:
        return ent[2]
    g = graph_from_dense(adj)
    _GRAPH_CACHE[key] = (weakref.ref(adj, lambda _r, k=key: _GRAPH_CACHE.pop(k, None)), adj._version, g)
    return g


def layer_fwd(m: torch.Tensor, wt: torch.Tensor, bias32: Optional[torch.Tensor], cdtype: torch.dtype, act: int):
    """Projection of an unfused layer: ``act(m W + b)`` from the aggregated rows ``m = A_hat x`` and the K-major weight
    ``wt [Dout,Din]``.  Returns ``(y, saved, split)``: ``saved`` is what :func:`layer_wgrad` reads, and ``split`` is None
    or the metadata of its fp32 split form.  In fp32 the projection runs on the tensor cores from split operands
    (ops.SplitRows); the split form of ``m`` is what the weight gradient reads, so it is saved instead of the fp32 rows
    (same bytes, one split per layer)."""
    if (cdtype == torch.float32 and ops.f32_tc(m.shape[0], m.shape[1], wt.shape[0])
            and ops.f32_tc(m.shape[0], wt.shape[0], m.shape[1])):
        m2 = ops.split_rows(m)
        return ops.linear_split(m2, ops.split_rows(wt), bias32, act), m2.data, (m2.amax, m2.rows, m2.cols)
    return ops.linear(m, wt, bias32, act=act), m, None


def layer_dy_split(dy: torch.Tensor, split):
    """The split form of ``dy`` when the layer ran split (shared by :func:`layer_wgrad` and :func:`layer_dgrad`)."""
    return ops.split_rows(dy) if split is not None else None


def layer_wgrad(saved: torch.Tensor, split, dy: torch.Tensor, dy2, bias_of: int):
    """``dW = (A_hat x)^T dy [Din,Dout]`` and ``db = colsum(dy)`` from :func:`layer_fwd`'s saved rows."""
    if split is not None:
        return ops.wgrad_split(ops.SplitRows(saved, *split), dy2, bias_of=bias_of)
    return ops.wgrad(saved, dy, bias_of=bias_of)


def layer_dgrad(dy: torch.Tensor, dy2, w: torch.Tensor) -> torch.Tensor:
    """``dy W^T`` with ``w [Din,Dout]`` (the input gradient before the adjoint aggregation)."""
    return ops.linear_split(dy2, ops.split_rows(w), None) if dy2 is not None else ops.linear(dy, w, None)


class _GCNLayerFn(torch.autograd.Function):
    """One graph convolution on packed rows: y = act((A_hat x) W + b).

    Forward  gcn.py:33-45; backward = what autograd derives for those lines:
    dW = (A_hat x)^T dy, db = colsum(dy), dx = A_hat^T (dy W^T)."""

    @staticmethod
    def forward(ctx, x, weight, bias, graph, cdtype, relu):
        xr = ops.as_rows(x, cdtype)
        m = ops.aggregate(xr, graph, mode=0)                               # A_hat x          [N,Din]
        wt = ops.cast_weight(weight, cdtype, transpose=True)               # [Dout,Din], K-major
        b32 = bias.detach().float().contiguous() if bias is not None else None
        y, m, ctx.split = layer_fwd(m, wt, b32, cdtype, L.ACT_RELU if relu else L.ACT_NONE)
        ctx.set_materialize_grads(False)
        ctx.graph, ctx.cdtype, ctx.relu, ctx.has_bias = graph, cdtype, relu, bias is not None
        ctx.x_dtype = x.dtype
        ctx.save_for_backward(m, weight, y if relu else None)
        return y

    @staticmethod
    def backward(ctx, dy):
        if dy is None:
            return None, None, None, None, None, None
        m, weight, y = ctx.saved_tensors
        graph, cdtype = ctx.graph, ctx.cdtype
        if ctx.relu:
            dy = dy * (y > 0)
        dyr = ops.as_rows(dy, cdtype)
        dW = db = dx = None
        dy2 = layer_dy_split(dyr, ctx.split)
        if ctx.needs_input_grad[1] or ctx.has_bias:
            dW, db = layer_wgrad(m, ctx.split, dyr, dy2, bias_of=2 if ctx.has_bias else 0)   # [Din,Dout], [Dout]
        if ctx.needs_input_grad[0]:
            w = ops.cast_weight(weight, cdtype, transpose=False)           # [Din,Dout] = B operand of dy W^T
            dx = ops.aggregate(layer_dgrad(dyr, dy2, w), graph, mode=1,
                               out_dtype=ctx.x_dtype if ctx.x_dtype in L.DTYPES else cdtype)
            if dx.dtype != ctx.x_dtype:
                dx = dx.to(ctx.x_dtype)
        return dx, dW, db, None, None, None


def gcn_layer(x: torch.Tensor, graph: DepGraph, weight: torch.Tensor, bias: Optional[torch.Tensor],
              compute_dtype=torch.float32, relu: bool = False) -> torch.Tensor:
    """Functional form on packed rows ``x [N,Din]`` -> ``[N,Dout]`` (compute dtype)."""
    return _GCNLayerFn.apply(x, weight, bias, graph, _compute_dtype(compute_dtype), relu)


class GraphConvolution(nn.Module):
    """Signature-compatible replacement of models/gcn.py:9-45.

    ``opt`` is accepted and ignored exactly as the reference ignores it
    (gcn.py:14); two optional attributes are read from it when present:
    ``opt.edg_dtype`` ('f32' default -- matches the reference to 1e-5 -- or 'bf16')
    and ``opt.edg_relu`` (default False: the reference applies no non-linearity,
    gcn.py:19 is dead code)."""

    def __init__(self, in_features, out_features, opt=None, bias=True, compute_dtype=None, relu=None):
        super().__init__()
        self.in_features = in_features
        self.out_features = out_features
        # gcn.py:18-21 leaves these uninitialised until train.py:75-84 runs; give them the same
        # distributions so a model used without Instructor._reset_params is still sane.
        self.weight = nn.Parameter(torch.empty(in_features, out_features))
        self.nonlinearity = nn.Tanh()       # kept (unused) so module listings match gcn.py:19
        if bias:
            self.bias = nn.Parameter(torch.empty(out_features))
        else:
            self.register_parameter("bias", None)
        self.compute_dtype = _compute_dtype(compute_dtype if compute_dtype is not None
                                            else getattr(opt, "edg_dtype", "f32"))
        self.relu = bool(relu if relu is not None else getattr(opt, "edg_relu", False))
        self.reset_parameters()

    def reset_parameters(self):
        nn.init.xavier_uniform_(self.weight)                         # train.py:80-81
        if self.bias is not None:
            stdv = 1.0 / math.sqrt(self.bias.shape[0])               # train.py:83-84
            nn.init.uniform_(self.bias, -stdv, stdv)

    def forward(self, text, adj):
        """text [B,T,Din] float, adj [B,T,T] (dense 0/1, self loops included) or a
        :class:`DepGraph` with ``text`` already packed as [N,Din]."""
        if isinstance(adj, DepGraph):
            y = gcn_layer(text, adj, self.weight, self.bias, self.compute_dtype, self.relu)
            return y if y.dtype == text.dtype else y.to(text.dtype)
        if not text.is_cuda:
            raise L.EdgError("GraphConvolution runs on CUDA tensors only (there is no CPU path)")
        B, T, Din = text.shape
        graph = cached_graph_from_dense(adj)
        y = gcn_layer(text.reshape(B * T, Din), graph, self.weight, self.bias, self.compute_dtype, self.relu)
        y = y.reshape(B, T, self.out_features)
        return y if y.dtype == text.dtype else y.to(text.dtype)

    def extra_repr(self):
        return f"{self.in_features}, {self.out_features}, compute={self.compute_dtype}, relu={self.relu}"
