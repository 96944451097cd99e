"""The trigger-conditioned gated GCN block as one module (reference: the inline
block every ``bert_amir*`` model repeats; canonical copy BertAmir55.forward,
models/bert_amir5.py:615-648, parameters :559-572).

``GatedGCNStack.forward`` computes, on packed rows and hand-written sm_100a kernels,

    a      = x[trigger row]                                   (:604-605, :615-618)
    g_l    = gate_l(a)                       l = 1..L         (:621-622, dropout p = 0)
    h_l    = gc_l(h_{l-1}, A),  h_0 = x      (ungated chain)  (:626, :639)
    xy     = sum_{l<l'} mean_b <max_t h_1*g_l, max_t h_1*g_l'> (:627-638)
    x_out  = g_L * h_L;  pooled = max_t x_out                 (:639-640)
    logits = logits_fn(a, pooled)            (host torch: self.dense(cat[...]), :643)
    scores = <logits, fc(cat[x_out, a])>     (collapsed: x_out . v_b + c_b)  (:645-646)
    kl     = mean_b sum_t softmax(scores) * softmax(float(dist))             (:648)

and the matching backward pass, as ONE autograd node.  At L = 2 this is exactly the
reference block.  CUDA only; no fallback.
"""
from __future__ import annotations

import contextlib
import os
from collections import namedtuple
from typing import Callable, List, Optional, Sequence

import torch
import torch.nn as nn

from . import _lib as L
from . import gcn, ops
from .gcn import GraphConvolution, _compute_dtype
from .graph import DepGraph, TriggerPairs

# name -> (leading Sigmoid?, Linears per gate, each followed by a Sigmoid); SURVEY 8a variant matrix
GATE_ARCHS = {
    "sig-2": (True, 2),     # BertAmir52/53/54/55   bert_amir5.py:562-571
    "2": (False, 2),        # BertAmir5/51          bert_amir5.py:27-30
    "3": (False, 3),        # BertAmir/BertAmir4    bert_amir.py:31-36
    "sig-3": (True, 3),     # BertAmir2             bert_amir.py:180-187
}



def _chain_ok(cd: torch.dtype, D: int, n_gates: int, gate_linears: int) -> bool:
    """The fused gate-MLP kernel (``edg_mlp_chain``) covers bf16, D <= 320, <= 4 gates, <= 3 Linears per gate;
    everything else runs one ``edg_linear`` per layer."""
    return (cd == torch.bfloat16 and 16 <= D <= ops.MLP_CHAIN_MAX_D and n_gates <= ops.MLP_CHAIN_MAX_GROUPS
            and gate_linears <= ops.MLP_CHAIN_MAX_STAGES)

# Two-stream overlap inside the autograd node (EDG_OVERLAP=0 disables it).  The gate MLPs (64 CTAs, latency-bound)
# and the view pooling are independent of the aggregate -> projection chain until their results meet, so they are
# enqueued on a side stream forked from / joined into the caller's stream with events; under CUDA-graph capture
# the fork/join become parallel branches of the graph.  Discipline that keeps the caching allocator safe without
# record_stream: the side stream always waits for the caller's current position before it starts, and the caller's
# stream always joins the side stream before the node returns.
_OVERLAP = os.environ.get("EDG_OVERLAP", "1") != "0"
_SIDE_STREAMS = {}
# SMs the input-gradient projection uses while the bucket all-reduce (grad_bucket_hook) runs next to it: the rest is
# what the collective's CTAs get
_BUCKET_LINEAR_SMS = 148 - int(os.environ.get("EDG_ALLREDUCE_SMS", "32"))

# The fused layer kernel (edg_gcn_layer: projection + tree aggregation + max-pool in one launch, both directions).
# EDG_FUSED=0 keeps the unfused aggregate -> linear -> pool kernels (bring-up / A-B timing).
_FUSED = os.environ.get("EDG_FUSED", "1") != "0"


def _dropout_seed(device) -> torch.Tensor:
    """The gate-dropout seed of one forward pass: a DEVICE int64 scalar drawn from torch's CUDA generator, so a captured
    CUDA graph draws fresh masks on every replay and ``torch.manual_seed`` makes them reproducible."""
    return torch.randint(0, 2 ** 62, (1,), dtype=torch.int64, device=device)


def _fused_plan(cfg, cd, D, graph, drop_p):
    """(tile_rows, plan) when the whole GCN chain can run on ``edg_gcn_layer``: bf16, no ReLU, no gate dropout, no
    BertAmir54 head on unpaired batches (their fused backward enters the chain through ``edg_head_du``, which has no
    sigmoid form; the pairs backward materialises d h_L whatever the head), every sentence fits a tile.  Otherwise None
    (the unfused kernels cover everything)."""
    fc_sig_unpaired = cfg["fc_sigmoid"] and cfg.get("pairs") is None
    if not _FUSED or cd != torch.bfloat16 or cfg["relu"] or drop_p > 0 or fc_sig_unpaired or cfg.get("view_len") is not None:
        return None
    rows = ops.fused_tile_rows(D, D)
    if rows <= 0:
        return None
    plan = graph.tile_plan(rows)
    return None if plan is None else (rows, plan)


def _masked_view_pool(h, graph: DepGraph, gates: torch.Tensor, view_len: torch.Tensor):
    """The two view pools of BertAmir / BertAmir2 (bert_amir.py:141-142, :282-283): ``masked_fill(mask, -1e12)`` before
    ``torch.max``, with ``mask`` = zeros then ones (data_utils.py:463-464), i.e. only the first ``view_len[b]`` rows of
    sentence b take part.  Runs the ordinary pooling kernel on a graph of 2B sentences (prefix, masked rest, prefix, ...)
    and keeps the prefixes; a sentence with nothing unmasked pools to the fill value and routes no gradient."""
    V, B, D = gates.shape
    sp = graph.sent_ptr.long()
    vl = torch.minimum(view_len.to(device=sp.device, dtype=torch.int64).clamp_min(0), sp[1:] - sp[:-1])
    sp2 = torch.empty(2 * B + 1, dtype=torch.int32, device=sp.device)
    sp2[0::2] = sp.int()
    sp2[1::2] = (sp[:-1] + vl).int()
    rs = graph.row_sent.long()
    local = torch.arange(graph.n_rows, device=sp.device) - sp[rs]
    rs2 = (2 * rs + (local >= vl[rs]).long()).int()
    g2 = DepGraph(sp2, graph.row_ptr, graph.col, rs2, 2 * B, graph.n_rows, graph.max_len)
    gg = gates.repeat_interleave(2, dim=1).contiguous()
    pooled, arg = ops.pool_fwd(h, g2, gg)
    pooled, arg = pooled[:, 0::2].contiguous(), arg[:, 0::2].contiguous()
    empty = (vl == 0)[None, :, None]
    return torch.where(empty, torch.full_like(pooled, -1e12), pooled), torch.where(empty, torch.full_like(arg, -1), arg)


def _side_stream(device: torch.device) -> "torch.cuda.Stream":
    idx = torch.device(device).index if torch.device(device).index is not None else torch.cuda.current_device()
    st = _SIDE_STREAMS.get(idx)
    if st is None:
        st = torch.cuda.Stream(device=idx)
        _SIDE_STREAMS[idx] = st
    return st


class _Side:
    """``with side.region():`` runs the body on the side stream after everything enqueued so far on the caller's
    stream; ``side.join()`` makes the caller's stream wait for all side work.  Disabled = plain in-order code."""

    def __init__(self, enabled: bool, device):
        self.enabled = enabled
        if enabled:
            self.main = torch.cuda.current_stream(device)
            self.side = _side_stream(device)
        self.dirty = False

    def region(self):
        if not self.enabled:
            return contextlib.nullcontext()
        self.side.wait_stream(self.main)
        self.dirty = True
        return torch.cuda.stream(self.side)

    def join(self):
        if self.enabled and self.dirty:
            self.main.wait_stream(self.side)
            self.dirty = False


def _check_head_leaves(logits: torch.Tensor, inner, declared) -> None:
    """``logits_fn`` may only depend on its two arguments and on the parameters passed as ``head_params``: anything else
    would silently train with a zero gradient (the block is one autograd node; the head's graph lives inside it)."""
    ok = {id(t) for t in inner} | {id(t) for t in declared}
    seen, todo = set(), [logits.grad_fn]
    while todo:
        fn = todo.pop()
        if fn is None or fn in seen:
            continue
        seen.add(fn)
        var = getattr(fn, "variable", None)
        if var is not None and var.requires_grad and id(var) not in ok:
            raise L.EdgError("logits_fn depends on a trainable tensor that was not passed in head_params "
                             f"(shape {tuple(var.shape)}): its gradient would be lost")
        todo.extend(f for f, _ in fn.next_functions)


StackOutput = namedtuple("StackOutput", ["logits", "xy", "kl", "scores", "pooled", "x_out", "pooled_arg", "view_arg"])


def make_gate(D: int, arch: str) -> nn.Sequential:
    lead, gate_linears = GATE_ARCHS[arch]
    mods: List[nn.Module] = [nn.Sigmoid()] if lead else []
    for _ in range(gate_linears):
        mods += [nn.Linear(D, D), nn.Sigmoid()]
    return nn.Sequential(*mods)


def _f32(t):
    return None if t is None else t.detach().float().contiguous()


def _x_rows(ctx, x: torch.Tensor, D: int, cd: torch.dtype) -> torch.Tensor:
    """x is [N, D], or the whole padded allocation [N, pitch >= D] (then dx comes back in the same dense layout and
    autograd can keep it without a copy): the compute-dtype rows, with what :func:`_dx_like_x` needs kept on ``ctx``."""
    ctx.x_padded, ctx.x_cols, ctx.x_dtype = x.shape[1] != D, x.shape[1], x.dtype
    return ops.as_rows(x[:, :D] if ctx.x_padded else x, cd)


def _dx_like_x(ctx, dx: torch.Tensor) -> torch.Tensor:
    """dx in the caller's layout: with a padded x, the whole [N, pitch] allocation (padding columns are finite)."""
    if ctx.x_padded:
        N, D = dx.shape
        dx = dx.as_strided((N, dx.stride(0)), (dx.stride(0), 1))
        if dx.shape[1] != ctx.x_cols:
            full = torch.zeros((N, ctx.x_cols), dtype=dx.dtype, device=dx.device)
            full[:, :D] = dx[:, :D]
            dx = full
    return dx if dx.dtype == ctx.x_dtype else dx.to(ctx.x_dtype)


def _param_groups(params, n_layers: int, gate_linears: int):
    """The block's parameter inputs -> (per layer (weight, bias), per gate per Linear (weight, bias) gate by gate,
    fc.weight, fc.bias)."""
    o = 2 * n_layers
    gate_p = [(params[k], params[k + 1]) for k in range(o, o + 2 * n_layers * gate_linears, 2)]
    return [(params[2 * l], params[2 * l + 1]) for l in range(n_layers)], gate_p, params[-2], params[-1]


def _unpack(params, cfg):
    """The Function's parameter inputs (the block's, then the classifier head's, whose gradients backward returns) ->
    (the block's parameters, GCN (weight, bias) per layer, gate (weight, bias) per Linear, fc.weight, fc.bias, w_t,
    w_n).  w_t / w_n are every compute-dtype weight copy of the step, transposed and in the same orientation (forward
    and backward operands), cast in one launch: the GCN layers' first, then the gates' in ``gate_p`` order."""
    n_head = cfg["n_head"]
    params = params[:len(params) - n_head] if n_head else params
    gcn_p, gate_p, fc_w, fc_b = _param_groups(params, cfg["L"], cfg["gate_linears"])
    flat_w = [w for (w, _) in gcn_p] + [w for (w, _) in gate_p]
    casted = ops.cast_weights_batch([(w, True) for w in flat_w] + [(w, False) for w in flat_w], cfg["cdtype"])
    nW = len(flat_w)
    return params, gcn_p, gate_p, fc_w, fc_b, casted[:nW], casted[nW:]


def _gates_fwd(s0, gate_p, w_n, gates: torch.Tensor, cd: torch.dtype, use_chain: bool):
    """The gate MLPs (bert_amir5.py:562-571) on ``s0 [M,D]``, the trigger rows after the leading Sigmoid of the
    architectures that have one: gate g's last Sigmoid writes ``gates[g]`` (fp32 ``[L,M,D]``).  ``gate_p`` / ``w_n``:
    the gates' parameters and same-orientation weights, gate by gate.  Returns per gate the inputs of its Linears."""
    Lyr, M, D = gates.shape
    n = len(gate_p) // Lyr
    saved = []
    if use_chain:
        # every Linear+Sigmoid of every gate in ONE launch (activation tile resident in shared memory)
        stages = []
        for g in range(Lyr):
            acts, st = [s0], []
            for i in range(n):
                last = i == n - 1
                out = gates[g] if last else ops.alloc_rows(M, D, cd, s0.device)
                st.append(dict(w=w_n[g * n + i], bias=_f32(gate_p[g * n + i][1]), out=out))
                if not last:
                    acts.append(out)
            stages.append(st)
            saved.append(acts)
        ops.mlp_chain(0, [s0] * Lyr, stages, M, D)
        return saved
    for g in range(Lyr):
        s, acts = s0, [s0]
        for i in range(n):
            last = i == n - 1                                           # nn.Linear [out,in] is K-major
            s = ops.linear(s, w_n[g * n + i], _f32(gate_p[g * n + i][1]), act=L.ACT_SIGMOID,
                           out_dtype=torch.float32 if last else cd, out=gates[g] if last else None)
            if not last:
                acts.append(s)
        saved.append(acts)
    return saved


def _gates_bwd(gates, dgates, saved, gate_p, w_t, lead: bool, cd: torch.dtype, use_chain: bool, grad_hook):
    """Backward of :func:`_gates_fwd` from the complete ``dgates``.  Returns ``(da_gate [M,D] or None, da_extra [L,M,D]
    or None, the gate parameters' gradients in parameter order)``: the gates' input gradients come back summed
    (``da_gate``, per-layer kernels) or as one slab per gate (``da_extra``, summed where it is consumed)."""
    Lyr, M, D = gates.shape
    n = len(gate_p) // Lyr
    dev = gates.device
    grads: List[Optional[torch.Tensor]] = [None] * (2 * len(gate_p))

    def put(g, i, dW, db):
        w, b = gate_p[g * n + i]
        grads[2 * (g * n + i)], grads[2 * (g * n + i) + 1] = dW.to(w.dtype), db.to(b.dtype)

    # the last Sigmoid of every gate in one launch (gates / dgates are [V*M, D] row blocks)
    dz_all = ops.sigmoid_bwd(gates.view(Lyr * M, D), dgates.view(Lyr * M, D), cd)
    da_gate = da_extra = None
    if use_chain:
        # d z chain of every gate in ONE launch, then every weight gradient in batched launches
        da_extra = torch.empty((Lyr, M, D), dtype=torch.float32, device=dev)
        dz_in = [[None] * n for _ in range(Lyr)]          # gradient at the pre-activation output of Linear i
        stages = []
        for g in range(Lyr):
            acts = saved[g]
            dz_in[g][n - 1] = dz_all[g * M:(g + 1) * M]
            st = []
            for i in range(n - 1, -1, -1):
                wt = w_t[g * n + i]                                     # [in,out]: row n = input column n
                if i > 0:
                    out = ops.alloc_rows(M, D, cd, dev)
                    dz_in[g][i - 1] = out
                    st.append(dict(w=wt, y=acts[i], out=out))
                else:
                    st.append(dict(w=wt, y=acts[0] if lead else None, out=da_extra[g]))
            stages.append(st)
        ops.mlp_chain(1, [dz_in[g][n - 1] for g in range(Lyr)], stages, M, D)
        idx = [(g, i) for g in range(Lyr) for i in range(n)]
        for c0 in range(0, len(idx), 8):
            part = idx[c0:c0 + 8]
            dWs, dbs = ops.wgrad_batch([dz_in[g][i] for g, i in part], [saved[g][i] for g, i in part], bias_of=1)
            for (g, i), dW, db in zip(part, dWs, dbs):
                put(g, i, dW, db)
    else:
        for g in range(Lyr):
            acts = saved[g]
            dz = dz_all[g * M:(g + 1) * M]
            for i in range(n - 1, -1, -1):
                put(g, i, *ops.wgrad(dz, acts[i], bias_of=1))            # [out,in], [out]
                wt = w_t[g * n + i]                                      # [in,out]
                if i > 0:
                    dz = ops.sigmoid_bwd(acts[i], ops.linear(dz, wt, None), cd)
                elif lead:
                    ds = ops.linear(dz, wt, None)
                    if da_gate is None:
                        da_gate = ops.sigmoid_bwd(acts[0], ds, torch.float32,
                                                  out=torch.empty((M, D), dtype=torch.float32, device=dev))
                    else:
                        ops.sigmoid_bwd(acts[0], ds, torch.float32, out=da_gate, accumulate=True)
                else:
                    dlast = ops.linear(dz, wt, None, out_dtype=torch.float32)
                    da_gate = dlast if da_gate is None else da_gate + dlast
    grad_hook(grads)
    return da_gate, da_extra, grads


def _head_fwd(ctx, a_raw, pooled, a_fc, fc_w, fc_b, hmax=None, gate=None):
    """Classifier head and the per-row operands of the collapsed scores, [v_b | va_b] = logits_b @ fc.weight and
    c_b = a_b . va_b + logits_b . fc.bias  (= logits_b . (Wfc[:, D:] a_b + bfc), SURVEY A9), in ONE launch
    (``edg_block_head_fwd``).  ``logits_fn`` is the model's own dense head (host torch, :643): it runs first under
    autograd and the launch takes its logits.  A head.DenseHead (= the reference's nn.Linear on cat[a, pooled]) runs
    inside the launch: no inner autograd graph, its weight and bias are head_params[0:2].  ``pooled`` None: pooled =
    gate * hmax (written by the launch for a DenseHead).  Returns (logits, v, c, pooled); what :func:`_head_bwd` reads
    stays on ``ctx``."""
    cfg = ctx.cfg
    dense = cfg.get("dense_head") is not None
    a_leaf = p_leaf = lg = w = bias = p = g = None
    if dense:
        hp = cfg["head_params"]
        w, bias = hp[0], hp[1] if len(hp) > 1 else None
        p, g = (hmax, gate) if pooled is None else (pooled, None)
    else:
        if pooled is None:
            pooled = gate * hmax
        with torch.enable_grad():
            a_leaf = a_raw.detach().requires_grad_(True)
            p_leaf = pooled.detach().requires_grad_(True)
            logits = cfg["logits_fn"](a_leaf, p_leaf)
        if logits.requires_grad and cfg["grad_enabled"]:
            _check_head_leaves(logits, (a_leaf, p_leaf), cfg["head_params"])
        lg = logits.detach().float().contiguous()
    n_head = w.shape[0] if dense else lg.shape[1]
    if n_head != fc_w.shape[0]:
        # the scores are <logits, fc(...)>: both heads have to give the same classes
        raise L.EdgError(f"logits_fn gives {n_head} classes, the stack's fc head {fc_w.shape[0]} (n_classes)")
    p_out, lg, v, c = ops.block_head_fwd(a_raw, a_fc, p, g, w, bias, _f32(fc_w), _f32(fc_b), logits=lg)
    if dense:
        pooled, logits = p_out, lg
    ctx.head = (a_leaf, p_leaf, logits, lg, a_raw, v)
    # (detached alias: `pooled` itself is an output of this node, and an output stored on its own node is a reference
    # cycle that keeps the whole graph -- and its AccumulateGrad nodes with their stream -- alive until the cyclic GC)
    ctx.pooled_head = pooled.detach() if dense else None
    return logits, v, c, pooled


def _head_bwd(ctx, g_logits, g_pooled, dvc, fc_w, fc_b, side: Optional[_Side], grad_hook):
    """Backward of :func:`_head_fwd`.  ``dvc = (d v, d c, scale)`` when the scores carry gradient (else None).  ONE
    launch (``edg_block_head_bwd``) gives d logits (``g_logits`` plus the fc's terms) and d a -- and for a DenseHead d
    pooled -- then every parameter gradient of the fc and of a DenseHead comes from one partial launch plus one
    reduction (``edg_block_head_wgrad``).  A torch head runs its own autograd graph on that d logits for its share of
    d a, d pooled and its parameters' gradients.  With ``side``, the parameter gradients (which nothing downstream
    waits for) run in ``side``'s region, where ``grad_hook`` receives them; with ``side=None`` they run inline and the
    caller hands them on.  Returns (d a or None, d pooled or None, d fc.weight, d fc.bias, head parameter
    gradients)."""
    cfg = ctx.cfg
    a_leaf, p_leaf, logits, lg, a_raw, v = ctx.head
    dense = cfg.get("dense_head") is not None
    hp = cfg["head_params"]
    region = side.region if side is not None else contextlib.nullcontext
    d_fcw = d_fcb = None
    g_lg = g_logits.float() if g_logits is not None else None
    head_grads: List[Optional[torch.Tensor]] = [None] * ctx.n_head
    da_k, gp_total = None, g_pooled
    # (a torch head without scores gradient: d logits is g_logits itself, nothing for the kernels to add)
    if dvc is not None or (dense and g_lg is not None):
        a_fc = ctx.fc_sig[2] if ctx.fc_sig else a_raw
        dv, dc, scale = dvc if dvc is not None else (None, None, None)
        w = hp[0] if dense else None
        # for a DenseHead d a and d pooled leave with everything else that flows into a / pooled already added
        g_lg, da_k, dp_k = ops.block_head_bwd(lg, a_raw, a_fc, bool(ctx.fc_sig), w, _f32(fc_w), _f32(fc_b), dv, dc,
                                              scale, g_lg, g_pooled if dense else None)
        if dense:
            gp_total = dp_k
        with region():
            d_hw, d_hb, d_fcw, d_fcb = ops.block_head_wgrad(lg, g_lg if dense else None, a_raw, a_fc,
                                                            ctx.pooled_head, dv, dc, scale,
                                                            want_bias=dense and len(hp) > 1)
            if d_fcw is not None:
                d_fcw, d_fcb = d_fcw.to(fc_w.dtype), d_fcb.to(fc_b.dtype)
                if side is not None:
                    grad_hook([d_fcw, d_fcb])
            if dense:
                if hp[0].requires_grad:
                    head_grads[0] = d_hw.to(hp[0].dtype)
                if len(hp) > 1 and hp[1].requires_grad:
                    head_grads[1] = d_hb.to(hp[1].dtype)
                if side is not None:
                    grad_hook([g for g in head_grads if g is not None and g.dtype == torch.float32])
    if dense:
        return da_k, gp_total, d_fcw, d_fcb, head_grads
    # ---- a torch head's own backward: d a, d pooled, and .grad of the parameters it closes over
    ga_head = gp_head = None
    if g_lg is not None and logits.requires_grad:
        cap = [(i, p) for i, p in enumerate(hp) if p.requires_grad]
        res = torch.autograd.grad([logits], [a_leaf, p_leaf] + [p for _, p in cap], [g_lg.to(logits.dtype)],
                                  allow_unused=True, retain_graph=True)
        ga_head, gp_head = res[0], res[1]
        for (i, _), g in zip(cap, res[2:]):
            head_grads[i] = g
        if side is not None:
            grad_hook([g for g in head_grads if g is not None and g.dtype == torch.float32])
    if da_k is not None:
        ga_head = da_k if ga_head is None else ga_head.float() + da_k
    if gp_head is not None:
        gp_total = gp_head.float() if gp_total is None else gp_total + gp_head.float()
    return ga_head, gp_total, d_fcw, d_fcb, head_grads


def _layer_fwd(h, wt, b, graph: DepGraph, cd: torch.dtype, relu: bool, fused, want_pool: bool):
    """One layer of the GCN chain -> (h_l, saved rows, split metadata, column maxima, their rows).  ``fused``: one
    ``edg_gcn_layer`` launch, h_l = A^ (h_{l-1} W_l) + b_l with the column maxima of every sentence (and their first
    rows) from the epilogue when ``want_pool`` -- the aggregated rows and the pooling passes never touch HBM.
    Otherwise aggregate -> projection (:func:`gcn.layer_fwd`), with no maxima."""
    if fused is not None:
        rows, plan = fused
        h, hm, ha, _ = ops.gcn_layer(h, wt, _f32(b), graph, 0, plan, rows, want_pool=want_pool)
        return h, None, None, hm, ha
    m = ops.aggregate(h, graph, mode=0)
    h, m, split = gcn.layer_fwd(m, wt, _f32(b), cd, L.ACT_RELU if relu else L.ACT_NONE)
    return h, m, split, None, None


def _unfused_layer_bwd(ctx, l: int, dh, hs, ms, params, grads_out, grad_hook):
    """Layer l of the unfused chain backward from d h_l: the ReLU mask, the weight gradient (handed to ``grad_hook``)
    and d h_l W_l^T, which the caller aggregates with A^T."""
    w, b = params[2 * l], params[2 * l + 1]
    if ctx.cfg["relu"]:
        dh = ops.as_rows(dh * (hs[l] > 0), ctx.cfg["cdtype"])
    split = ctx.ms_split[l]
    dh2 = gcn.layer_dy_split(dh, split)                                 # shared by dW and the input gradient
    dW, db = gcn.layer_wgrad(ms[l], split, dh, dh2, bias_of=2)
    grads_out[2 * l], grads_out[2 * l + 1] = dW.to(w.dtype), db.to(b.dtype)
    grad_hook(grads_out[2 * l:2 * l + 2])
    return gcn.layer_dgrad(dh, dh2, ctx.w_n[l])                          # w_n[l] [in,out] = B operand of dh W^T


def _fused_chain_bwd(ctx, du, db_next, xr, hs, params, grads_out, grad_hook, patch=None, patch_ready=None):
    """The fused chain backward from du_L = A^T dh_L and db_L.  With u_l = h_{l-1} W_l and h_l = A^ u_l + b_l:
    db_l = colsum(dh_l), du_l = A^T dh_l, dW_l = h_{l-1}^T du_l, dh_{l-1} = du_l W_l^T.  One fused launch per layer
    produces du_{l-1} = A^T (du_l W_l^T + views patch) and the column sums of its argument (= db_{l-1}); neither
    dh_{l-1} nor the aggregated rows exist in HBM.  ``patch`` (the views' share of d h_1) enters the layer-1 launch,
    after ``patch_ready`` when given.  Returns du_1 once the weight gradient of layer 1 is handed to ``grad_hook``:
    dx = du_1 W_1^T is the caller's."""
    rows, plan = ctx.fused
    graph = ctx.cfg["graph"]
    for l in range(len(hs) - 1, -1, -1):
        w, b = params[2 * l], params[2 * l + 1]
        dW, _ = ops.wgrad(hs[l - 1] if l > 0 else xr, du, bias_of=0)
        grads_out[2 * l], grads_out[2 * l + 1] = dW.to(w.dtype), db_next.to(b.dtype)
        grad_hook(grads_out[2 * l:2 * l + 2])
        if l > 0:
            if l == 1 and patch_ready is not None:
                torch.cuda.current_stream(xr.device).wait_event(patch_ready)
            du, _, _, db_next = ops.gcn_layer(du, ctx.w_n[l], None, graph, 1, plan, rows,
                                              patch=patch if l == 1 else None, want_colsum=True)
    return du


class _GatedStackFn(torch.autograd.Function):
    """inputs: x, then per layer (weight, bias), then per gate per Linear (weight, bias),
    then fc.weight, fc.bias.  ``cfg`` carries the non-tensor arguments."""

    @staticmethod
    def forward(ctx, cfg, x, aspect, *params):
        graph: DepGraph = cfg["graph"]
        cd: torch.dtype = cfg["cdtype"]
        Lyr, lead, D = cfg["L"], cfg["lead"], cfg["D"]
        B = graph.n_graphs
        xr = _x_rows(ctx, x, D, cd)
        params, gcn_p, gate_p, fc_w, fc_b, w_t, w_n = _unpack(params, cfg)
        ctx.w_t, ctx.w_n = w_t, w_n
        # ---- trigger vector and the gate MLPs (bert_amir5.py:615-622)
        gated = cfg["gated"]
        drop_p, seed = (cfg["drop_p"], cfg["seed"]) if gated else (0.0, None)
        h1m = None
        ctx.ext_aspect = aspect is not None
        if aspect is not None:
            # the trigger vector comes from the caller (BertAmir / BertAmir2: max-pool of the LSTM output over the
            # trigger's word pieces, bert_amir.py:118) instead of the trigger row of x (bert_amir5.py:615-618)
            a_raw = aspect.detach().float().contiguous()
            s0 = ops.as_rows(torch.sigmoid(a_raw) if lead else a_raw, cd)
        side = _Side(_OVERLAP and gated, x.device)
        if aspect is None:
            with side.region():                   # the gather feeds the gate MLPs only: it runs on their (side) stream
                a_raw, s0 = ops.trigger_gather(xr, graph, cfg["anchor"], lead)
        # ungated ablation (BertAmir55NoGate, bert_amir5.py:731-749): x = gc2(gc1(x)), out = max_t x, xy = 0.0; the same
        # kernels run with a unit gate
        gates = (torch.empty if gated else torch.ones)((Lyr, B, D), dtype=torch.float32, device=x.device)
        ctx.use_chain = gated and _chain_ok(cd, D, Lyr, cfg["gate_linears"])
        with side.region():                       # overlaps the first aggregate -> projection below
            gate_saved = _gates_fwd(s0, gate_p, w_n[Lyr:], gates, cd, ctx.use_chain) if gated else []
        # ---- ungated GCN chain (bert_amir5.py:626, :639; gcn.py:33-45); after layer 1 the gated views of h_1 and
        # the diversity term (:627-638) go to the side stream (behind the gate MLPs) while layers 2.. run here
        h = xr
        ms, hs, ms_split = [], [], []
        v_pooled = v_arg = v_hmax = None
        xy = torch.zeros((), dtype=torch.float32, device=x.device)
        fused = _fused_plan(cfg, cd, D, graph, drop_p)
        ctx.fused = fused
        for l, (_, b) in enumerate(gcn_p):
            views_here = l == 0 and gated
            h, m, split, hm, ha = _layer_fwd(h, w_t[l], b, graph, cd, cfg["relu"], fused, views_here or l == Lyr - 1)
            ms.append(m)
            ms_split.append(split)
            hs.append(h)
            if views_here and fused is not None:
                v_hmax = hm
                v_arg = ha.unsqueeze(0).expand(Lyr, B, D)     # positive gates: the views share their arg-max row
                if Lyr > 1:
                    with side.region():
                        v_pooled = gates * hm.unsqueeze(0)    # max_t (h_t g) = g max_t h_t for g > 0
                        xy = ops.diversity_fwd(v_pooled)
            elif views_here:
                with side.region():
                    if drop_p > 0:
                        # gate dropout (:624-625): view v sees h_1 under the per-token mask of gate v
                        h1m = [ops.dropout_rows(hs[0], seed, v, drop_p) for v in range(Lyr)]
                        v_pooled = torch.empty((Lyr, B, D), dtype=torch.float32, device=x.device)
                        v_arg = torch.empty((Lyr, B, D), dtype=torch.int32, device=x.device)
                        for v in range(Lyr):
                            pv, av = ops.pool_fwd(h1m[v], graph, gates[v:v + 1])
                            v_pooled[v], v_arg[v] = pv[0], av[0]
                    elif cfg.get("view_len") is not None:
                        v_pooled, v_arg = _masked_view_pool(hs[0], graph, gates, cfg["view_len"])
                    else:
                        v_pooled, v_arg = ops.pool_fwd(hs[0], graph, gates)
                    if Lyr > 1:
                        xy = ops.diversity_fwd(v_pooled)
        side.join()                                # gates (and the views) are complete from here on
        # ---- output pooling (:639-640); under gate dropout x_out = gate_L * (h_L * mask_L / (1-p))
        gL = gates[Lyr - 1]
        if fused is not None:
            hL, hmaxL, p_arg = hs[-1], hm, ha
            pooled = None                              # gL * hmaxL, from the head launch; the arg-max rows came with the maxima
        else:
            hL = ops.dropout_rows(hs[-1], seed, Lyr - 1, drop_p) if drop_p > 0 else hs[-1]
            hmaxL = None
            pooled, p_arg = ops.pool_fwd(hL, graph, gL.unsqueeze(0))
            pooled, p_arg = pooled[0], p_arg[0]
        # ---- classifier head (:643) and the scores' per-sentence operands
        ctx.set_materialize_grads(False)          # unused outputs arrive as None, not zero tensors
        ctx.cfg = cfg
        fc_sig = cfg["fc_sigmoid"]
        # BertAmir54: fc = Sequential(Sigmoid, Linear) (:464-465): the scores read z = sigmoid(x_out) (materialised
        # rows, unit gate) and sigmoid(a); everything downstream is the same kernels
        a_fc = torch.sigmoid(a_raw) if fc_sig else a_raw
        logits, v, c, pooled = _head_fwd(ctx, a_raw, pooled, a_fc, fc_w, fc_b, hmaxL, gL)
        # ---- importance scores and the softmax product (:645-648)
        # (also d kl/d v, d kl/d c per unit gradient: saves the backward pass one sweep over h_L)
        if fc_sig:
            z = ops.gate_rows(hL, graph, gL, cd, act=L.ACT_SIGMOID)
            ones = torch.ones((B, D), dtype=torch.float32, device=x.device)
            scores, kl_b, kl, dvu, dcu = ops.scores_kl_fwd(z, graph, ones, v, c, cfg["dist"], want_units=True)
            ctx.fc_sig = (z, ones, a_fc)
        else:
            if fused is not None:
                scores, kl_b, kl, dvu, dcu, uu, sfu = ops.scores_kl_fwd(hL, graph, gL, v, c, cfg["dist"],
                                                                        want_units=True, want_rows=True)
                ctx.kl_rows = (uu, sfu)
            else:
                scores, kl_b, kl, dvu, dcu = ops.scores_kl_fwd(hL, graph, gL, v, c, cfg["dist"], want_units=True)
            ctx.fc_sig = None
        ctx.kl_units = (dvu, dcu)
        x_out = ops.gate_rows(hL, graph, gL, cd) if cfg["return_x_out"] else None
        ctx.drop = (drop_p, seed, h1m, hL) if drop_p > 0 else None
        ctx.gate_saved = gate_saved
        ctx.n_params = len(params)
        ctx.n_head = cfg["n_head"]
        ctx.v_hmax = v_hmax
        ctx.hmaxL = hmaxL
        ctx.ms_split = ms_split
        if fused is not None and v_arg is not None:
            v_arg = v_arg.contiguous()
        ctx.save_for_backward(xr, gates, v_pooled, v_arg, p_arg, scores, kl_b, *ms, *hs, *params)
        # arg-max rows (global row ids), like the indices torch.max returns at :635-636/:640
        if v_arg is None:
            v_arg = torch.empty((0,), dtype=torch.int32, device=x.device)
        ctx.mark_non_differentiable(p_arg, v_arg)
        return logits.detach(), xy, kl, scores, pooled, x_out, p_arg, v_arg

    @staticmethod
    def backward(ctx, g_logits, g_xy, g_kl, g_scores, g_pooled, g_xout, _g_parg=None, _g_varg=None):
        cfg = ctx.cfg
        graph: DepGraph = cfg["graph"]
        cd: torch.dtype = cfg["cdtype"]
        Lyr, dist = cfg["L"], cfg["dist"]
        saved = ctx.saved_tensors
        xr, gates, v_pooled, v_arg, p_arg, scores, kl_b = saved[:7]
        ms = saved[7:7 + Lyr]
        hs = saved[7 + Lyr:7 + 2 * Lyr]
        params = saved[7 + 2 * Lyr:]
        _, gate_p, fc_w, fc_b = _param_groups(params, Lyr, cfg["gate_linears"])
        B, N, D = graph.n_graphs, graph.n_rows, xr.shape[1]
        dev = xr.device
        v = ctx.head[5]
        gL = gates[Lyr - 1]
        drop = ctx.drop
        hL = drop[3] if drop else hs[-1]          # under gate dropout the block ran on the masked rows of h_L
        g_xy, g_kl, g_scores, g_pooled = _f32(g_xy), _f32(g_kl), _f32(g_scores), _f32(g_pooled)
        if g_xout is not None:
            g_xout = ops.as_rows(g_xout, cd)
        need_scores = g_kl is not None or g_scores is not None
        grad_hook = cfg.get("grad_hook") or (lambda ts: None)
        bucket_hook = cfg.get("bucket_hook")
        gated = cfg["gated"]
        views_active = g_xy is not None and Lyr > 1 and gated
        dgates = torch.empty((Lyr, B, D), dtype=torch.float32, device=dev)
        side = _Side(_OVERLAP and gated, dev)
        # (the unfused path keeps ONE edg_views_bwd launch at layer 1: issuing its dgates half early on the side
        # stream was measured slower, 0.989 vs 0.965 ms/step -- the two halves re-read the same [B,D] arrays)
        fused = ctx.fused
        # ---- d v, d c: the per-unit gradients of the forward sweep times d kl, or (when scores itself carries
        # gradient) pass A over h_L; then the fc and classifier heads
        dvc = None
        if need_scores:
            if g_scores is None:
                dvc = (ctx.kl_units[0], ctx.kl_units[1], g_kl)
            else:
                rows_s, gate_s = (ctx.fc_sig[0], ctx.fc_sig[1]) if ctx.fc_sig else (hL, gL)
                _, _, dv_in, dc_in = ops.head_bwd(rows_s, graph, gate_s, v, dist, scores, kl_b, g_kl, g_scores,
                                                  None, None, None, want_dh=False, want_dv=True)
                dvc = (dv_in, dc_in, None)
        ga_head, gp_total, d_fcw, d_fcb, head_grads = _head_bwd(ctx, g_logits, g_pooled, dvc, fc_w, fc_b, side,
                                                                grad_hook)
        gp_total = gp_total.contiguous() if gp_total is not None else None
        # ---- pass B over h_L: dh_L, dgate_L
        if not views_active and Lyr > 1:
            dgates[:Lyr - 1].zero_()                                  # no diversity gradient: the other gates get none
        dgL = dgates[Lyr - 1]
        du_top = db_top = None
        if fused is not None and g_xout is None:
            # top of the chain straight in aggregated form: du_L = A^T dh_L, db_L, d gate_L from [N]- and [B,D]-sized
            # inputs only (h_L is not read again, dh_L never exists)
            uu, sfu = ctx.kl_rows
            du_top, db_top, _ = ops.head_du(uu, g_kl if need_scores else None, g_scores, gL, v, gp_total, p_arg, sfu,
                                            ctx.hmaxL, graph, fused[1], want_dgate=True, dgate_out=dgL)
            if g_scores is not None:
                # scores itself carries gradient: d gate_L also needs sum_t g_scores_t h_t -- one sweep over h_L
                _, _, dv_s, _ = ops.head_bwd(hL, graph, gL, v, dist, scores, kl_b, None, g_scores, None, None, None,
                                             want_dh=False, want_dv=True)
                dgL.add_(torch.where(gL != 0, dv_s * v / gL, torch.zeros_like(gL)))
            dh = None
        elif ctx.fc_sig and need_scores:
            # scores branch on z = sigmoid(x_out): d z (unit gate), through the sigmoid, then into the x_out path
            z, ones, _ = ctx.fc_sig
            dz, _, _, _ = ops.head_bwd(z, graph, ones, v, dist, scores, kl_b, g_kl, g_scores, None, None, None,
                                       want_dh=True, want_dv=False)
            dxo = ops.sigmoid_bwd(z, dz, cd)
            if g_xout is not None:
                dxo = ops.as_rows(dxo + g_xout, cd)
            dh, _, _, _ = ops.head_bwd(hL, graph, gL, None, dist, None, kl_b, None, None, gp_total, p_arg, dxo,
                                       want_dh=True, want_dv=False, dgate_out=dgL)
        else:
            dh, _, _, _ = ops.head_bwd(hL, graph, gL, v if need_scores else None, dist,
                                       scores if need_scores else None, kl_b, g_kl, g_scores, gp_total, p_arg, g_xout,
                                       want_dh=True, want_dv=False, dgate_out=dgL)
        if drop:
            dh = ops.dropout_rows(dh, drop[1], Lyr - 1, drop[0])      # d h_L = d (h_L * mask / (1-p)) * mask / (1-p)
        grads_out: List[Optional[torch.Tensor]] = [None] * ctx.n_params
        o = 2 * Lyr

        # ---- gate MLP backward (bert_amir5.py:562-571): needs the complete dgates, nothing else of the GCN chain;
        # it runs on the side stream next to the GCN chain backward
        def gate_backward():
            da_g, da_x, gg = _gates_bwd(gates, dgates, ctx.gate_saved, gate_p, ctx.w_t[Lyr:], cfg["lead"], cd,
                                        ctx.use_chain, grad_hook)
            grads_out[o:o + len(gg)] = gg
            return da_g, da_x

        da_gate = da_extra = None
        if fused is not None:
            if du_top is not None:
                du, db_next = du_top, db_top
            else:                                 # a direct gradient on x_out came in: dh_L exists, aggregate it
                db_next = ops.colsum(dh)
                du = ops.aggregate(dh, graph, mode=1)
            patch = None
            patch_ready = None
            if gated:
                # side stream, behind edg_head_du (which wrote d gate_L): the views' share of d gates / the patch for d h_1,
                # then the gate MLPs' backward; this stream goes straight on to the weight gradient of layer L and only
                # waits for the patch where it is consumed (the layer-1 launch)
                with side.region():
                    if views_active:
                        patch = (ops.views_bwd_hmax(ctx.v_hmax, gates, g_xy, dgates, acc_view=Lyr - 1), v_arg[0])
                        if side.enabled:
                            patch_ready = torch.cuda.Event()
                            patch_ready.record(side.side)
                    da_gate, da_extra = gate_backward()     # dgates are complete from here on
            du = _fused_chain_bwd(ctx, du, db_next, xr, hs, params, grads_out, grad_hook, patch, patch_ready)
            wk = ctx.w_n[0]                                                 # [in,out] = B operand of du W^T
            if bucket_hook is not None:
                # every parameter gradient of the block exists now (the gate MLPs' come from the side stream): hand
                # them to the all-reduce and let it run NEXT to the input-gradient projection, which leaves it SMs
                side.join()
                grads_out[-2], grads_out[-1] = d_fcw, d_fcb
                n_out = len(grads_out)
                reduced = bucket_hook(list(grads_out) + list(head_grads))
                grads_out[:] = reduced[:n_out]
                head_grads = list(reduced[n_out:])
                d_fcw, d_fcb = grads_out[-2], grads_out[-1]
                with ops.sm_budget(_BUCKET_LINEAR_SMS):
                    dh = ops.linear(du, wk, None)
            else:
                dh = ops.linear(du, wk, None)
        else:
            for l in range(Lyr - 1, -1, -1):
                if l == 0 and views_active and drop:
                    # every view pooled its own masked copy of h_1: route per view, then mask the row gradient again
                    dp = (g_xy / B) * (v_pooled.sum(0, keepdim=True) - v_pooled)              # d xy / d pooled_v  (:638)
                    for vi in range(Lyr):
                        tmp = ops.alloc_rows(N, D, cd, dev, zero=True)
                        ops.views_bwd(v_pooled[vi:vi + 1], v_arg[vi:vi + 1], gates[vi:vi + 1], drop[2][vi], None,
                                      dp[vi:vi + 1].contiguous(), tmp, dgates[vi:vi + 1], acc_view=0 if vi == Lyr - 1 else -1)
                        ops.dropout_rows(tmp, drop[1], vi, drop[0], out=dh, accumulate=True)
                elif l == 0 and views_active:
                    # gated views of h_1 feed xy (:627-638): add their gradient to d h_1 before leaving layer 1
                    ops.views_bwd(v_pooled, v_arg, gates, hs[0], g_xy, None, dh, dgates, acc_view=Lyr - 1)
                if l == 0 and gated:
                    with side.region():               # dgates are complete from here on
                        da_gate, da_extra = gate_backward()
                dm = _unfused_layer_bwd(ctx, l, dh, hs, ms, params, grads_out, grad_hook)
                dh = ops.aggregate(dm, graph, mode=1)
        dx = dh
        side.join()
        da = ga_head.float() if ga_head is not None else None
        if da_extra is not None and ctx.ext_aspect:   # the caller gets d aspect as a tensor: sum the gates' slabs here
            da_gate, da_extra = (da_extra.sum(0) if da_extra.shape[0] > 1 else da_extra[0]), None
        if da_gate is not None:
            da = da_gate if da is None else da + da_gate
        d_aspect = None
        if da is not None or da_extra is not None:
            if ctx.ext_aspect:
                d_aspect = da
            else:
                ops.trigger_scatter_add(da, graph, cfg["anchor"], dx, extra=da_extra)
        grads_out[-2], grads_out[-1] = d_fcw, d_fcb
        return (None, _dx_like_x(ctx, dx), d_aspect) + tuple(grads_out) + tuple(head_grads)


class _GatedPairsFn(torch.autograd.Function):
    """The block for (sentence, trigger) pairs (``GatedGCNStack.forward(..., pairs=)``): the GCN chain runs once on the
    sentence rows, everything that depends on the trigger runs per pair.  Positive gates give
    ``max_t (h_t * g) = g * max_t h_t`` with a gate-independent arg-max row, so every per-pair pooled view is
    ``g_p * hmax[sentence(p)]``; only the scores / kl pass over the sentence's rows once per pair.  Same inputs as
    :class:`_GatedStackFn` (without ``aspect``)."""

    @staticmethod
    def forward(ctx, cfg, x, *params):
        graph: DepGraph = cfg["graph"]
        pairs: TriggerPairs = cfg["pairs"]
        cd: torch.dtype = cfg["cdtype"]
        Lyr, D, gated = cfg["L"], cfg["D"], cfg["gated"]
        S, P = graph.n_graphs, pairs.n_pairs
        xr = _x_rows(ctx, x, D, cd)
        params, gcn_p, gate_p, fc_w, fc_b, w_t, w_n = _unpack(params, cfg)
        ctx.w_t, ctx.w_n = w_t, w_n
        # ---- per pair: the trigger row of its sentence and the gate MLPs on P rows
        a_raw, s0 = ops.trigger_gather(xr, ops.PairRows(pairs), cfg["anchor"], cfg["lead"])
        gates = (torch.empty if gated else torch.ones)((Lyr, P, D), dtype=torch.float32, device=x.device)
        ctx.use_chain = gated and _chain_ok(cd, D, Lyr, cfg["gate_linears"])
        gate_saved = _gates_fwd(s0, gate_p, w_n[Lyr:], gates, cd, ctx.use_chain) if gated and P > 0 else []
        # gate dropout (pair_dropout=True): every pair pools and scores its own masked copy of the sentence rows, so the
        # per-sentence column maxima below are not used
        drop_p, seed = (cfg["drop_p"], cfg["seed"]) if gated else (0.0, None)
        # ---- the GCN chain once per sentence, with the column maxima of h_1 (views) and h_L (final pool)
        h = xr
        ms, hs, ms_split = [], [], []
        hmax1 = harg1 = hm = ha = None
        fused = _fused_plan(cfg, cd, D, graph, drop_p)
        ctx.fused = fused
        ones = None
        for l, (_, b) in enumerate(gcn_p):
            want_pool = ((l == 0 and gated) or l == Lyr - 1) and drop_p == 0
            h, m, split, hm, ha = _layer_fwd(h, w_t[l], b, graph, cd, cfg["relu"], fused, want_pool)
            if fused is None and want_pool:
                if ones is None:
                    ones = torch.ones((1, S, D), dtype=torch.float32, device=x.device)
                _, ha, hm = ops.pool_fwd(h, graph, ones, want_hmax=True)
                ha = ha[0]
            ms.append(m)
            ms_split.append(split)
            hs.append(h)
            if l == 0 and gated:
                hmax1, harg1 = hm, ha
        hmaxL, hargL = hm, ha
        ps = pairs.pair_sent.long()
        xy = torch.zeros((), dtype=torch.float32, device=x.device)
        v_arg = None
        gL = gates[Lyr - 1]
        hL = hs[-1]
        ctx.drop = None
        if drop_p > 0:
            # views: h_1 under the masks of streams 0..L-1; final pool and scores: h_L under stream L-1
            v_pooled, v_arg, v_mmax = ops.pool_drop_pairs(hs[0], graph, pairs, gates, seed, 0, drop_p)
            if Lyr > 1 and P > 0:
                xy = ops.diversity_fwd(v_pooled)
            pooled, p_arg, mmaxL = (t[0] for t in ops.pool_drop_pairs(hL, graph, pairs, gL.unsqueeze(0), seed, Lyr - 1,
                                                                      drop_p))
            ctx.drop = (drop_p, seed, v_pooled, v_mmax, v_arg.detach(), p_arg.detach(), mmaxL)
        else:
            if gated:
                v_arg = harg1[ps].unsqueeze(0).expand(Lyr, P, D).contiguous()
                if Lyr > 1 and P > 0:
                    xy = ops.diversity_fwd(gates * hmax1[ps].unsqueeze(0))     # views g_{v,p} * max_t h_1
            pooled = gL * hmaxL[ps]
            p_arg = hargL[ps]
        # ---- classifier head on [P,D], then the per-pair scores / kl over the sentence rows
        ctx.set_materialize_grads(False)
        ctx.cfg = cfg
        fc_sig = cfg["fc_sigmoid"]
        # BertAmir54 (pair_fc_sigmoid): the fc head reads sigmoid(a); the scores read z = sigmoid(g_p * h_t), which the
        # per-pair kernels form from each row as they read it (no z rows: ctx.fc_sig carries only sigmoid(a))
        a_fc = torch.sigmoid(a_raw) if fc_sig else a_raw
        ctx.fc_sig = (None, None, a_fc) if fc_sig else None
        logits, v, c, pooled = _head_fwd(ctx, a_raw, pooled, a_fc, fc_w, fc_b)
        if fc_sig:
            scores, kl_b, kl, dvu, dcu = ops.scores_kl_sig_pairs_fwd(hL, graph, pairs, gL, v, c, cfg["dist"],
                                                                     seed if drop_p > 0 else None, Lyr - 1, drop_p)
        elif drop_p > 0:
            scores, kl_b, kl, dvu, dcu = ops.scores_kl_drop_pairs_fwd(hL, graph, pairs, gL, v, c, cfg["dist"], seed,
                                                                      Lyr - 1, drop_p)
        else:
            scores, kl_b, kl, dvu, dcu = ops.scores_kl_pairs_fwd(hL, graph, pairs, gL, v, c, cfg["dist"])
        ctx.kl_units = (dvu, dcu)
        ctx.gate_saved = gate_saved
        ctx.n_params = len(params)
        ctx.n_head = cfg["n_head"]
        ctx.ms_split = ms_split
        ctx.pool_rows = (hmax1, harg1, hargL)
        ctx.save_for_backward(xr, gates, scores, kl_b, *ms, *hs, *params)
        if v_arg is None:
            v_arg = torch.empty((0,), dtype=torch.int32, device=x.device)
        ctx.mark_non_differentiable(p_arg, v_arg)
        return logits.detach(), xy, kl, scores, pooled, p_arg, v_arg

    @staticmethod
    def backward(ctx, g_logits, g_xy, g_kl, g_scores, g_pooled, _g_parg=None, _g_varg=None):
        cfg = ctx.cfg
        graph: DepGraph = cfg["graph"]
        pairs: TriggerPairs = cfg["pairs"]
        Lyr, dist = cfg["L"], cfg["dist"]
        saved = ctx.saved_tensors
        xr, gates, scores, kl_b = saved[:4]
        ms = saved[4:4 + Lyr]
        hs = saved[4 + Lyr:4 + 2 * Lyr]
        params = saved[4 + 2 * Lyr:]
        _, gate_p, fc_w, fc_b = _param_groups(params, Lyr, cfg["gate_linears"])
        P, D = pairs.n_pairs, xr.shape[1]
        dev = xr.device
        v = ctx.head[5]
        hmax1, harg1, hargL = ctx.pool_rows
        gL = gates[Lyr - 1]
        hL = hs[-1]
        g_xy, g_kl, g_scores, g_pooled = _f32(g_xy), _f32(g_kl), _f32(g_scores), _f32(g_pooled)
        need_scores = g_kl is not None or g_scores is not None
        grad_hook = cfg.get("grad_hook") or (lambda ts: None)
        gated = cfg["gated"]
        views_active = g_xy is not None and Lyr > 1 and gated
        dgates = torch.empty((Lyr, P, D), dtype=torch.float32, device=dev)
        drop = ctx.drop
        if drop:
            drop_p, seed, v_pooled, v_mmax, v_arg, p_arg, mmaxL = drop
        if ctx.fc_sig:
            # BertAmir54: through z = sigmoid(g_p * h_t) per (pair, row), masked as in the forward pass
            pool_seed = (p_arg, mmaxL, seed, Lyr - 1, drop_p) if drop else (hargL, None, None, 0, 0.0)

            def head_bwd(*a, **kw):
                return ops.head_bwd_sig_pairs(*a, *pool_seed, **kw)
        elif drop:
            # the head backward on every pair's masked rows of h_L (stream L-1), with the pair's own final-pool rows
            def head_bwd(*a, **kw):
                return ops.head_bwd_drop_pairs(*a, p_arg, mmaxL, seed, Lyr - 1, drop_p, **kw)
        else:
            def head_bwd(*a, **kw):
                return ops.head_bwd_pairs(*a, hargL, **kw)
        # ---- d v, d c (per pair), the fc head and the classifier head
        dvc = None
        if need_scores:
            if g_scores is None:
                dvc = (ctx.kl_units[0], ctx.kl_units[1], g_kl)
            else:
                _, _, dv_in, dc_in = head_bwd(hL, graph, pairs, gL, v, dist, scores, kl_b, g_kl, g_scores, None,
                                              want_dh=False)
                dvc = (dv_in, dc_in, None)
        ga_head, gp_total, d_fcw, d_fcb, head_grads = _head_bwd(ctx, g_logits, g_pooled, dvc, fc_w, fc_b, None, None)
        grad_hook([g for g in head_grads if g is not None and g.dtype == torch.float32])
        # ---- d h_L over the sentence rows (every pair of a sentence summed in pair order), d gate_L per pair
        if not views_active and Lyr > 1:
            dgates[:Lyr - 1].zero_()
        dh, _, _, _ = head_bwd(hL, graph, pairs, gL, v if need_scores else None, dist, scores if need_scores else None,
                               kl_b, g_kl, g_scores, gp_total.contiguous() if gp_total is not None else None,
                               want_dh=True, dgate_out=dgates[Lyr - 1])
        patch_val = None
        if views_active and drop:
            ops.views_bwd_drop_pairs(v_pooled, v_mmax, v_arg, gates, g_xy, graph, pairs, seed, drop_p, dgates=dgates,
                                     acc_view=Lyr - 1)
        elif views_active:
            patch_val = ops.views_bwd_hmax_pairs(hmax1, gates, g_xy, dgates, pairs, acc_view=Lyr - 1)
        grads_out: List[Optional[torch.Tensor]] = [None] * ctx.n_params
        o = 2 * Lyr
        # ---- gate MLPs (dgates complete)
        da_gate = da_extra = None
        if gated and P > 0:
            da_gate, da_extra, gg = _gates_bwd(gates, dgates, ctx.gate_saved, gate_p, ctx.w_t[Lyr:], cfg["lead"],
                                               cfg["cdtype"], ctx.use_chain, grad_hook)
            grads_out[o:o + len(gg)] = gg
        elif gated:                                # no pairs: the gate parameters get zero gradients
            for k in range(o, o + 2 * len(gate_p)):
                grads_out[k] = torch.zeros_like(params[k])
        # ---- the GCN chain backward on the sentence rows, exactly as for unpaired batches
        if ctx.fused is not None:
            patch = (patch_val, harg1) if patch_val is not None else None
            db_next = ops.colsum(dh)
            du = _fused_chain_bwd(ctx, ops.aggregate(dh, graph, mode=1), db_next, xr, hs, params, grads_out, grad_hook,
                                  patch)
            dh = ops.linear(du, ctx.w_n[0], None)
        else:
            for l in range(Lyr - 1, -1, -1):
                if l == 0 and views_active and drop:
                    # the views' share of d h_1: every pair's view arg-max rows under that view's mask
                    ops.views_bwd_drop_pairs(v_pooled, v_mmax, v_arg, gates, g_xy, graph, pairs, seed, drop_p, dh=dh)
                if l == 0 and patch_val is not None:
                    # the views' share of d h_1 at the sentences' arg-max rows ((row, column) targets are distinct):
                    # edg_views_bwd_parts with one unit view adds g_pooled = patch_val at arg
                    zero = torch.zeros((1, graph.n_graphs, D), dtype=torch.float32, device=dev)
                    ops.views_bwd(zero, harg1.unsqueeze(0), zero + 1.0, hs[0], None, patch_val.unsqueeze(0), dh, None,
                                  parts=1)
                dh = ops.aggregate(_unfused_layer_bwd(ctx, l, dh, hs, ms, params, grads_out, grad_hook), graph, mode=1)
        dx = dh
        # ---- d x at the trigger rows: the head's and the gate MLPs' d a of every pair, in pair order
        da = ga_head.float() if ga_head is not None else None
        if da_gate is not None:
            da = da_gate if da is None else da + da_gate
        if (da is not None or da_extra is not None) and P > 0:
            ops.trigger_scatter_add_pairs(da, pairs, cfg["anchor"], dx, extra=da_extra)
        grads_out[-2], grads_out[-1] = d_fcw, d_fcb
        grad_hook([g for g in (d_fcw, d_fcb) if g is not None])
        return (None, _dx_like_x(ctx, dx)) + tuple(grads_out) + tuple(head_grads)


class GatedGCNStack(nn.Module):
    """Owns gc1..gcL, gate1..gateL and fc with the reference's parameter names
    (state-dict keys ``gc1.weight``, ``gate1.1.weight``, ``fc.0.weight`` ...,
    bert_amir5.py:559-572) and runs the whole block fused."""

    def __init__(self, hidden: int, n_layers: int = 2, n_classes: int = 2, gate_arch: str = "sig-2",
                 relu: bool = False, dropout: float = 0.0, compute_dtype="f32", gated: bool = True,
                 fc_sigmoid: bool = False, pair_dropout: bool = False, pair_fc_sigmoid: bool = False):
        super().__init__()
        if hidden % 4:
            raise ValueError("hidden size must be a multiple of 4 (16-byte fp32 rows)")
        self.hidden, self.n_layers, self.n_classes = hidden, n_layers, n_classes
        self.gate_arch = gate_arch
        self.gated = gated            # False = BertAmir55NoGate (gates constructed, as there, but unused: :672-681, :731-748)
        self.relu = relu
        self.dropout_p = dropout
        # train-mode gate dropout on the pairs= path (per-pair passes over the sentence rows instead of [P,D] products:
        # the caller asks for that cost explicitly); no effect without pairs, in eval mode, at p = 0 or ungated
        self.pair_dropout = pair_dropout
        # BertAmir54's sigmoid fc head on the pairs= path (every pair's z = sigmoid(g_p * h_t) formed in per-pair passes
        # over the sentence rows); no effect without fc_sigmoid or without pairs
        self.pair_fc_sigmoid = pair_fc_sigmoid
        self.compute_dtype = _compute_dtype(compute_dtype)
        for l in range(1, n_layers + 1):
            setattr(self, f"gc{l}", GraphConvolution(hidden, hidden, None, compute_dtype=self.compute_dtype))
            setattr(self, f"gate{l}", make_gate(hidden, gate_arch))
        # data parallelism: called inside the backward pass with every group of parameter gradients the moment it exists
        # (parallel.GradientAllReducer.hook all-reduces it in place while the layers below still run); None = single GPU
        self.grad_ready_hook = None
        # optional callable(list of gradient tensors or None) -> same list with the tensors it took replaced: called ONCE
        # per backward pass of the fused path, when every parameter gradient of the block exists and only the input
        # gradient is left to compute (parallel.GradientAllReducer.bucket packs them into one flat buffer and starts
        # its all-reduce, which then overlaps that last projection)
        self.grad_bucket_hook = None
        self.fc_sigmoid = fc_sigmoid
        if fc_sigmoid:                                                   # BertAmir54, bert_amir5.py:464-465 (keys fc.1.*)
            self.fc = nn.Sequential(nn.Sigmoid(), nn.Linear(2 * hidden, n_classes))
        else:
            self.fc = nn.Sequential(nn.Linear(2 * hidden, n_classes))    # bert_amir5.py:572

    def _flat_params(self) -> List[torch.Tensor]:
        ps: List[torch.Tensor] = []
        for l in range(1, self.n_layers + 1):
            gc = getattr(self, f"gc{l}")
            ps += [gc.weight, gc.bias]
        for l in range(1, self.n_layers + 1):
            for m in getattr(self, f"gate{l}"):
                if isinstance(m, nn.Linear):
                    ps += [m.weight, m.bias]
        ps += [self.fc[-1].weight, self.fc[-1].bias]
        return ps

    def forward(self, x: torch.Tensor, graph: DepGraph, anchor_index: torch.Tensor, dist_to_target: torch.Tensor,
                logits_fn: Callable[[torch.Tensor, torch.Tensor], torch.Tensor],
                head_params: Sequence[torch.Tensor] = (), return_x_out: bool = False,
                aspect: Optional[torch.Tensor] = None, view_len: Optional[torch.Tensor] = None,
                pairs: Optional[TriggerPairs] = None) -> StackOutput:
        """x [N,D] packed rows (or [B,T,D] with a dense-compat graph), graph, sentence-local
        trigger index [B], distances (packed [N] or [B,T] for a dense-compat graph; int32/int64),
        ``logits_fn(a [B,D], pooled [B,D]) -> [B,C]`` = the model's ``dense`` head (:643), and the
        parameters ``logits_fn`` closes over (so their gradients are delivered).

        ``aspect [B,D]`` (optional): the trigger vector, when the model computes it itself (BertAmir / BertAmir2 pool the
        LSTM output over the trigger's word pieces, bert_amir.py:118, :259) instead of taking the trigger row of ``x``;
        its gradient is returned through autograd.  ``view_len int [B]`` (optional): the two diversity pools only see the
        first ``view_len[b]`` rows of sentence b -- ``masked_fill(mask, -1e12)`` of bert_amir.py:141-142 with the
        reference's zeros-then-ones mask (``view_len = (mask == 0).sum(1)``); the final pool stays unmasked (:146).

        ``pairs`` (:class:`graph.TriggerPairs`, ``graph.pairs_from_ptr``): score every candidate trigger of a sentence
        from ONE pass of the GCN chain.  ``x [N,D]`` and ``graph`` then hold every sentence once; ``anchor_index [P]``
        and ``dist_to_target`` (per-pair packed, ``[pairs.n_pair_rows]``) are per (sentence, trigger) pair.  Every
        output is per pair -- ``logits [P,C]``, ``pooled [P,D]``, ``scores [n_pair_rows]``, ``pooled_arg [P,D]`` and
        ``view_arg [V,P,D]`` (global sentence rows) -- and ``xy`` / ``kl`` are means over the P pairs; ``logits_fn``
        receives ``[P,D]`` inputs.  The result equals the block run on the batch with each sentence repeated once per
        pair, ``dx`` being the sum over a sentence's pairs.  Valid only when ``x`` does not depend on the trigger
        (no trigger marker or position features upstream).  Train-mode gate dropout (``dropout > 0``) needs
        ``pair_dropout=True``: each pair then applies the masks the expanded batch would apply to its copy of the
        sentence (keyed on the per-pair packed row ``pairs.pair_row_ptr[p] + t``), so for the same
        ``last_dropout_seed`` the result equals the expanded run's, every pair with its own masks; the views and the
        final pool become per-pair passes over the sentence rows.  BertAmir54's head (``fc_sigmoid``) needs
        ``pair_fc_sigmoid=True``: each pair's scores then read ``sigmoid(g_p * h_t)``, formed per (pair, row) as the
        sentence rows are read (with or without ``pair_dropout``).  Not covered (``EdgError``): train-mode gate dropout
        without ``pair_dropout``, ``fc_sigmoid`` without ``pair_fc_sigmoid``, ``view_len``, ``aspect``,
        ``return_x_out`` and 3-D dense-compat ``x``."""
        if not x.is_cuda:
            raise L.EdgError("GatedGCNStack runs on CUDA tensors only (there is no CPU path)")
        if pairs is not None:
            return self._forward_pairs(x, graph, anchor_index, dist_to_target, logits_fn, head_params, return_x_out,
                                       aspect, view_len, pairs)
        drop_p, seed = 0.0, None
        if self.training and self.dropout_p > 0 and self.gated:
            # nn.Dropout on the broadcast gates (bert_amir5.py:624-625).  The seed is a DEVICE scalar drawn from
            # torch's CUDA generator, so a captured CUDA graph draws a fresh mask on every replay.
            drop_p = float(self.dropout_p)
            seed = _dropout_seed(x.device)
            self.last_dropout_seed = seed
        shape3 = None
        if x.dim() == 3:
            shape3 = x.shape
            x = x.reshape(-1, x.shape[-1])
        cfg = self._cfg(x, graph, anchor_index, dist_to_target.reshape(-1), logits_fn, head_params)
        cfg.update(bucket_hook=self.grad_bucket_hook, return_x_out=return_x_out, drop_p=drop_p, seed=seed,
                   view_len=view_len)
        logits, xy, kl, scores, pooled, x_out, p_arg, v_arg = _GatedStackFn.apply(cfg, x, aspect, *self._flat_params(),
                                                                                 *cfg["head_params"])
        if shape3 is not None:
            scores = scores.reshape(shape3[0], shape3[1])
            if x_out is not None:
                x_out = x_out.reshape(shape3)
        return StackOutput(logits, xy, kl, scores, pooled, x_out, p_arg, v_arg)

    def _cfg(self, x, graph, anchor_index, dist, logits_fn, head_params) -> dict:
        """The non-tensor arguments both block Functions read (``dist`` flat)."""
        if dist.dtype not in (torch.int32, torch.int64):
            dist = dist.long()
        if x.shape[-1] != self.hidden and x.shape[-1] != ops.row_pitch(self.hidden, x.dtype):
            raise L.EdgError(f"expected {self.hidden} feature columns (or the padded pitch), got {x.shape[-1]}")
        lead, gate_linears = GATE_ARCHS[self.gate_arch]
        from .head import DenseHead
        dense_head = logits_fn if isinstance(logits_fn, DenseHead) and logits_fn.fusable(self.hidden) else None
        if isinstance(logits_fn, DenseHead):        # its parameters are the head parameters: nothing to declare
            head_params = [p for p in (logits_fn.weight, logits_fn.bias) if p is not None]
        head_params = list(head_params)
        return dict(graph=graph, cdtype=self.compute_dtype, D=self.hidden, dense_head=dense_head, L=self.n_layers,
                    gate_linears=gate_linears, lead=lead, anchor=anchor_index.to(torch.int32).contiguous(),
                    dist=dist.contiguous(), logits_fn=logits_fn, head_params=head_params, n_head=len(head_params),
                    grad_enabled=torch.is_grad_enabled(), grad_hook=self.grad_ready_hook, relu=self.relu,
                    gated=self.gated, fc_sigmoid=self.fc_sigmoid)

    def _forward_pairs(self, x, graph, anchor_index, dist_to_target, logits_fn, head_params, return_x_out, aspect,
                       view_len, pairs: TriggerPairs) -> StackOutput:
        declined = []
        drop = self.training and self.dropout_p > 0 and self.gated
        if drop and not self.pair_dropout:
            declined.append("train-mode gate dropout (p > 0) unless GatedGCNStack(pair_dropout=True)")
        if self.fc_sigmoid and not self.pair_fc_sigmoid:
            declined.append("fc_sigmoid unless GatedGCNStack(pair_fc_sigmoid=True)")
        if view_len is not None:
            declined.append("view_len")
        if aspect is not None:
            declined.append("aspect")
        if return_x_out:
            declined.append("return_x_out")
        if x.dim() != 2:
            declined.append("3-D dense-compat x")
        if self.grad_bucket_hook is not None:
            declined.append("grad_bucket_hook (sharded grouped batches)")
        if declined:
            raise L.EdgError("pairs= does not cover: " + ", ".join(declined))
        drop_p, seed = 0.0, None
        if drop:
            drop_p = float(self.dropout_p)
            seed = _dropout_seed(x.device)
            self.last_dropout_seed = seed
        if pairs.n_sentences != graph.n_graphs:
            raise L.EdgError(f"pairs were built for {pairs.n_sentences} sentences, the graph has {graph.n_graphs}")
        if x.shape[0] != graph.n_rows:
            raise L.EdgError(f"x has {x.shape[0]} rows, the graph {graph.n_rows} (pass each sentence once)")
        if anchor_index.numel() != pairs.n_pairs:
            raise L.EdgError(f"expected {pairs.n_pairs} anchors (one per pair), got {anchor_index.numel()}")
        dist = dist_to_target.reshape(-1)
        if dist.numel() != pairs.n_pair_rows:
            raise L.EdgError(f"dist_to_target must be per-pair packed ({pairs.n_pair_rows} entries), got {dist.numel()}")
        cfg = self._cfg(x, graph, anchor_index, dist, logits_fn, head_params)
        cfg.update(pairs=pairs, drop_p=drop_p, seed=seed)
        logits, xy, kl, scores, pooled, p_arg, v_arg = _GatedPairsFn.apply(cfg, x, *self._flat_params(),
                                                                           *cfg["head_params"])
        return StackOutput(logits, xy, kl, scores, pooled, None, p_arg, v_arg)
