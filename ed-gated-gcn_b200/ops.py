"""Thin tensor-level wrappers over the C ABI: allocate outputs with torch (device
memory + stream plumbing), pass raw pointers / leading dimensions to libedgcn.

Row matrices are 2-D views ``[N, D]`` of a ``[N, ld]`` allocation with
``ld = round_up(D, 16 bytes)`` so every row starts 16-byte aligned (128-bit
loads, TMA global-stride rule).  Padding columns are always finite.
"""
from __future__ import annotations

from typing import Optional

import torch

from . import _lib as L


def _round_up(a: int, b: int) -> int:
    return (a + b - 1) // b * b


def row_pitch(D: int, dtype: torch.dtype) -> int:
    return _round_up(D, 16 // torch.empty((), dtype=dtype).element_size())


def alloc_rows(N: int, D: int, dtype: torch.dtype, device, zero: bool = False, min_ld: int = 0) -> torch.Tensor:
    ld = max(row_pitch(D, dtype), min_ld)
    base = (torch.zeros if zero else torch.empty)((max(N, 1), ld), dtype=dtype, device=device)
    return base[:N, :D]


def as_rows(t: torch.Tensor, dtype: torch.dtype) -> torch.Tensor:
    """Return ``t`` as an aligned 2-D row matrix of ``dtype`` (repacked only if needed)."""
    if not t.is_cuda:
        raise L.EdgError("libedgcn takes CUDA tensors only (there is no CPU path)")
    assert t.dim() == 2
    es = t.element_size()
    ok = (t.dtype == dtype and t.stride(1) == 1 and (t.stride(0) * es) % 16 == 0 and t.data_ptr() % 16 == 0
          and t.stride(0) >= t.shape[1])
    if ok:
        return t
    out = alloc_rows(t.shape[0], t.shape[1], dtype, t.device, zero=True)
    out.copy_(t)
    return out


def ld(t: torch.Tensor) -> int:
    return t.stride(0)


def _f32c(t: torch.Tensor) -> torch.Tensor:
    t = t.detach()
    return t if (t.dtype == torch.float32 and t.is_contiguous()) else t.float().contiguous()


# ---------------------------------------------------------------------------
def aggregate(x: torch.Tensor, graph, mode: int, out_dtype: Optional[torch.dtype] = None) -> torch.Tensor:
    N, D = x.shape
    # the kernel walks 16-byte chunks of the INPUT dtype, so the output pitch must cover the same columns
    out = alloc_rows(N, D, out_dtype or x.dtype, x.device, min_ld=row_pitch(D, x.dtype))
    L.call("edg_aggregate", L.ptr(x), L.dt(x), ld(x), L.ptr(out), L.dt(out), ld(out), N, D,
           L.ptr(graph.row_ptr), L.ptr(graph.col), mode, L.ptr(graph.sent_ptr), L.ptr(graph.row_sent),
           graph.n_graphs, graph.max_len, L.stream())
    return out


class sm_budget:
    """``with ops.sm_budget(n):`` the persistent projection kernel launched inside uses at most ``n`` SMs
    (``edg_set_sm_budget``), leaving the rest to a collective running next to it."""

    def __init__(self, n: int):
        self.n = int(n)

    def __enter__(self):
        self.prev = int(L.load().edg_set_sm_budget(self.n))
        return self

    def __exit__(self, *exc):
        L.load().edg_set_sm_budget(self.prev)
        return False


class SplitRows:
    """An fp32 row matrix in the split form the fp32-parity tensor-core GEMMs read (``edg_split_f16``):
    ``data`` fp16 ``[rows, 2 * round_up(cols, 64)]`` = ``[hi | lo]`` of ``x * 2^k``, ``amax`` the device scalar the
    power-of-two scale is derived from."""
    __slots__ = ("data", "amax", "rows", "cols")

    def __init__(self, data, amax, rows, cols):
        self.data, self.amax, self.rows, self.cols = data, amax, rows, cols

    @property
    def shape(self):
        return (self.rows, self.cols)


F32_TC_MIN_ROWS = 1024      # below this the FFMA kernels win (five launches against one)


def f32_tc(rows: int, K: int, Nout: int) -> bool:
    """Whether an fp32 ``[rows, K] x [Nout, K]^T`` product runs on the tensor cores in split form
    (``EDG_F32_TC=0`` keeps the FFMA kernels: bring-up switch)."""
    import os
    if os.environ.get("EDG_F32_TC", "1") == "0" or rows < F32_TC_MIN_ROWS:
        return False
    if rows * ((max(K, Nout) + 63) // 64) * 16 >= 2 ** 31:      # edg_split_f16 counts elements in 32 bits
        return False
    return bool(L.load().edg_linear_split_ok(int(K), int(Nout)))


def split_rows(x: torch.Tensor) -> SplitRows:
    """``edg_split_f16``: fp32 ``[rows, cols]`` -> :class:`SplitRows` (two launches: max |x|, then hi / lo)."""
    x = as_rows(x, torch.float32)
    rows, cols = x.shape
    pitch = int(L.load().edg_split_pitch(cols))
    data = torch.empty((max(rows, 1), pitch), dtype=torch.float16, device=x.device)
    amax = torch.empty((1,), dtype=torch.float32, device=x.device)
    L.call("edg_split_f16", L.ptr(x), ld(x), rows, cols, L.ptr(data), pitch, L.ptr(amax), L.stream())
    return SplitRows(data, amax, rows, cols)


def linear_split(a: SplitRows, w: SplitRows, bias: Optional[torch.Tensor], act: int = L.ACT_NONE,
                 out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """``act(a @ w.T + bias)`` in fp32 from split operands (``edg_linear_split``); ``w`` is ``[Nout, K]``."""
    M, K = a.shape
    Nout = w.rows
    assert w.cols == K
    if out is None:
        out = alloc_rows(M, Nout, torch.float32, a.data.device)
    L.call("edg_linear_split", L.ptr(a.data), a.data.stride(0), L.ptr(a.amax), M, K, L.ptr(w.data), w.data.stride(0),
           L.ptr(w.amax), Nout, L.ptr(bias), act, L.ptr(out), ld(out), L.stream())
    return out


def wgrad_split(a: SplitRows, b: SplitRows, bias_of: int = 0):
    """``a.T @ b`` in fp32 (+ column sums of a (1) or b (2)) from split operands (``edg_wgrad_split``)."""
    R, K1 = a.shape
    K2 = b.cols
    assert b.rows == R
    dev = a.data.device
    dW = torch.empty((K1, K2), dtype=torch.float32, device=dev)
    db = torch.empty((K1 if bias_of == 1 else K2,), dtype=torch.float32, device=dev) if bias_of else None
    nbytes = L.load().edg_wgrad_split_workspace(R, K1, K2)
    ws = torch.empty((nbytes + 255) // 4, dtype=torch.float32, device=dev)
    L.call("edg_wgrad_split", L.ptr(a.data), a.data.stride(0), L.ptr(a.amax), K1, L.ptr(b.data), b.data.stride(0),
           L.ptr(b.amax), K2, R, L.ptr(dW), K2, L.ptr(db), bias_of, L.ptr(ws), ws.numel() * 4, L.stream())
    return dW, db


def linear(a: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor], act: int = L.ACT_NONE,
           out_dtype: Optional[torch.dtype] = None, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """``act(a @ w.T + bias)`` with ``w`` given as ``[Nout, K]`` (K contiguous).  fp32 operands with enough rows go
    through the split tensor-core path (:func:`f32_tc`)."""
    M, K = a.shape
    Nout = w.shape[0]
    assert w.shape[1] == K and a.dtype == w.dtype
    if (a.dtype == torch.float32 and (out_dtype or a.dtype) == torch.float32 and (out is None or out.dtype == torch.float32)
            and f32_tc(M, K, Nout)):
        return linear_split(split_rows(a), split_rows(w), bias, act, out)
    if out is None:
        out = alloc_rows(M, Nout, out_dtype or a.dtype, a.device)
    L.call("edg_linear", L.ptr(a), L.dt(a), ld(a), M, K, L.ptr(w), ld(w), Nout, L.ptr(bias), act,
           L.ptr(out), L.dt(out), ld(out), L.stream())
    return out


FUSED_MAX_SENTENCES = 6     # sentences per tile of edg_tile_plan (kFMaxSent in csrc/edg_gcn_fused.cu)


def fused_tile_rows(K: int, Nout: int) -> int:
    """Rows per tile the fused layer kernel supports for this shape (0: shape not covered)."""
    return int(L.load().edg_fused_tile_rows(K, Nout))


def gcn_layer(x: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor], graph, mode: int, plan, tile_rows: int,
              want_pool: bool = False, patch=None, want_colsum: bool = False):
    """``edg_gcn_layer``: ``A^ (x w.T) + bias`` (mode 0, optionally with the per-sentence column maxima
    ``hmax fp32 [B,Nout]`` / ``harg int32 [B,Nout]``) or ``A^T (x w.T + patch)`` (mode 1, optionally with the
    column sums of the un-aggregated rows).  ``w`` is ``[Nout, K]`` bf16, ``plan = graph.tile_plan(tile_rows)``.
    Returns ``(y, hmax, harg, colsum)``."""
    N, K = x.shape
    Nout = w.shape[0]
    assert x.dtype == torch.bfloat16 and w.dtype == torch.bfloat16 and w.shape[1] == K
    B = graph.n_graphs
    dev = x.device
    y = alloc_rows(N, Nout, torch.bfloat16, dev)
    hmax = torch.empty((B, Nout), dtype=torch.float32, device=dev) if want_pool else None
    harg = torch.empty((B, Nout), dtype=torch.int32, device=dev) if want_pool else None
    colsum = torch.empty((Nout,), dtype=torch.float32, device=dev) if want_colsum else None
    ws = torch.empty((148 * Nout,), dtype=torch.float32, device=dev) if want_colsum else None
    pv, pa = patch if patch is not None else (None, None)
    info, n_tiles = plan
    L.call("edg_gcn_layer", L.ptr(x), ld(x), N, K, L.ptr(w), ld(w), Nout, L.ptr(bias), int(mode), L.ptr(graph.row_ptr),
           L.ptr(graph.col), L.ptr(graph.sent_ptr), L.ptr(info), L.ptr(n_tiles), int(tile_rows), L.ptr(y), ld(y),
           L.ptr(hmax), L.ptr(harg), Nout, L.ptr(pv), L.ptr(pa), pv.stride(0) if pv is not None else 0, L.ptr(colsum), 0,
           L.ptr(ws), ws.numel() * 4 if ws is not None else 0, L.stream())
    return y, hmax, harg, colsum


def views_bwd_hmax(hmax: torch.Tensor, gates: torch.Tensor, g_xy, dgates: torch.Tensor, acc_view: int = -1) -> torch.Tensor:
    """Backward of the pooled views + diversity term from the column maxima: writes ``dgates`` and returns
    ``patch_val fp32 [B,D]`` (what the arg-max rows of d h_1 receive)."""
    V, B, D = gates.shape
    patch_val = torch.empty((B, D), dtype=torch.float32, device=hmax.device)
    L.call("edg_views_bwd_hmax", L.ptr(hmax), L.ptr(gates), L.ptr(g_xy), V, B, D, L.ptr(patch_val), D, L.ptr(dgates),
           int(acc_view), L.stream())
    return patch_val


def head_du(u_unit, g_kl, g_scores, gate, v, g_pooled, arg, sf_unit, hmax, graph, plan, want_dgate: bool = True,
            dgate_out: Optional[torch.Tensor] = None):
    """``edg_head_du``: ``du_L = A^T dh_L`` (bf16 rows), ``db_L`` and ``d gate_L`` from per-row scalars and
    per-sentence vectors only (see include/edgcn.h).  Returns ``(du, dbias, dgate)``."""
    B, D = gate.shape
    N = u_unit.shape[0]
    dev = gate.device
    du = alloc_rows(N, D, torch.bfloat16, dev)
    dbias = torch.empty((D,), dtype=torch.float32, device=dev)
    dgate = (dgate_out if dgate_out is not None else torch.empty((B, D), dtype=torch.float32, device=dev)) if want_dgate else None
    nbytes = L.load().edg_head_du_workspace(D)
    ws = torch.empty(nbytes // 4, dtype=torch.float32, device=dev)
    info, n_tiles = plan
    L.call("edg_head_du", L.ptr(u_unit), L.ptr(g_kl), L.ptr(g_scores), L.ptr(gate), L.ptr(v), L.ptr(g_pooled), L.ptr(arg),
           L.ptr(sf_unit), L.ptr(hmax), N, B, D, L.ptr(graph.row_ptr), L.ptr(graph.col), L.ptr(graph.sent_ptr), L.ptr(info),
           L.ptr(n_tiles), L.ptr(du), ld(du), L.ptr(dgate), L.ptr(dbias), L.ptr(ws), ws.numel() * 4, L.stream())
    return du, dbias, dgate


def wgrad(a: torch.Tensor, b: torch.Tensor, bias_of: int = 0):
    """``a.T @ b`` in fp32 (+ column sums of a (1) or b (2))."""
    R, K1 = a.shape
    K2 = b.shape[1]
    assert b.shape[0] == R and a.dtype == b.dtype
    if a.dtype == torch.float32 and f32_tc(R, K1, K2) and f32_tc(R, K2, K1):
        return wgrad_split(split_rows(a), split_rows(b), bias_of)
    dW = torch.empty((K1, K2), dtype=torch.float32, device=a.device)
    db = torch.empty((K1 if bias_of == 1 else K2,), dtype=torch.float32, device=a.device) if bias_of else None
    nbytes = L.load().edg_wgrad_workspace(R, K1, K2, L.dt(a))
    ws = torch.empty((nbytes + 255) // 4, dtype=torch.float32, device=a.device)
    L.call("edg_wgrad", L.ptr(a), ld(a), K1, L.ptr(b), ld(b), K2, L.dt(a), R, L.ptr(dW), K2, L.ptr(db), bias_of, 0,
           L.ptr(ws), ws.numel() * 4, L.stream())
    return dW, db


def wgrad_batch(a_list, b_list, bias_of: int = 0):
    """``a_i.T @ b_i`` (+ column sums) for several same-shaped bf16 problems in one launch.
    Returns ([dW_i], [db_i])."""
    import ctypes
    n = len(a_list)
    R, K1 = a_list[0].shape
    K2 = b_list[0].shape[1]
    dev = a_list[0].device
    lda, ldb = ld(a_list[0]), ld(b_list[0])
    for a, b in zip(a_list, b_list):
        assert a.shape == (R, K1) and b.shape == (R, K2) and ld(a) == lda and ld(b) == ldb and a.dtype == b.dtype
    dW = torch.empty((n, K1, K2), dtype=torch.float32, device=dev)
    nb = K1 if bias_of == 1 else K2
    db = torch.empty((n, nb), dtype=torch.float32, device=dev) if bias_of else None
    nbytes = L.load().edg_wgrad_batch_workspace(n, R, K1, K2)
    ws = torch.empty((nbytes + 255) // 4, dtype=torch.float32, device=dev)
    P = ctypes.c_void_p * n
    L.call("edg_wgrad_batch", n, P(*[L.ptr(a) for a in a_list]), lda, K1, P(*[L.ptr(b) for b in b_list]), ldb, K2,
           L.dt(a_list[0]), R, P(*[L.ptr(dW[i]) for i in range(n)]), K2,
           P(*[L.ptr(db[i]) for i in range(n)]) if bias_of else None, bias_of, L.ptr(ws), ws.numel() * 4, L.stream())
    return [dW[i] for i in range(n)], ([db[i] for i in range(n)] if bias_of else [None] * n)


MLP_CHAIN_MAX_D = 320
MLP_CHAIN_MAX_GROUPS = 4
MLP_CHAIN_MAX_STAGES = 3


def mlp_chain(mode: int, a0_list, stages, M: int, D: int) -> None:
    """One launch for ``len(a0_list)`` chains of Linear layers (see ``edg_mlp_chain``).
    ``stages[g][s]`` = dict(w=, bias=None, y=None, out=None) of tensors."""
    import ctypes
    n_groups, n_stages = len(a0_list), len(stages[0])
    arr = (L.ChainStage * (n_groups * n_stages))()
    for g in range(n_groups):
        for s_i, st in enumerate(stages[g]):
            e = arr[g * n_stages + s_i]
            w, y, out, bias = st["w"], st.get("y"), st.get("out"), st.get("bias")
            e.w, e.ldw = L.ptr(w), ld(w)
            e.bias = L.ptr(bias)
            e.y, e.ldy = (L.ptr(y), ld(y)) if y is not None else (None, 0)
            e.out, e.ldo = (L.ptr(out), ld(out)) if out is not None else (None, 0)
            e.out_dtype = L.dt(out) if out is not None else 0
    P = ctypes.c_void_p * n_groups
    L.call("edg_mlp_chain", mode, n_groups, n_stages, P(*[L.ptr(a) for a in a0_list]), ld(a0_list[0]), arr, M, D,
           L.stream())


def cast_weight(w: torch.Tensor, dtype: torch.dtype, transpose: bool) -> torch.Tensor:
    """fp32 master weight ``[R,C]`` -> compute-dtype ``[R,C]`` or ``[C,R]`` row matrix."""
    w = w.detach()
    if w.dtype != torch.float32 or not w.is_contiguous():
        w = w.float().contiguous()
    R, C = w.shape
    ro, co = (C, R) if transpose else (R, C)
    out = alloc_rows(ro, co, dtype, w.device)
    L.call("edg_cast_2d", L.ptr(w), w.stride(0), R, C, L.ptr(out), L.dt(out), ld(out), int(transpose), L.stream())
    return out


def cast_weights_batch(items, dtype: torch.dtype):
    """``items`` = [(fp32 weight [R,C], transpose?)]: all compute-dtype copies in one kernel launch.
    Returns the row matrices in the same order (views of one flat allocation)."""
    import ctypes
    n = len(items)
    ws = []
    for w, _ in items:
        w = w.detach()
        if w.dtype != torch.float32 or not w.is_contiguous():
            w = w.float().contiguous()
        ws.append(w)
    shapes = [((w.shape[1], w.shape[0]) if tr else tuple(w.shape)) for w, (_, tr) in zip(ws, items)]
    lds = [row_pitch(co, dtype) for _, co in shapes]
    sizes = [_round_up(ro * l, 64) for (ro, _), l in zip(shapes, lds)]       # keep every slice 128-byte aligned
    flat = torch.empty(sum(sizes), dtype=dtype, device=ws[0].device)
    outs, off = [], 0
    for (ro, co), l, sz in zip(shapes, lds, sizes):
        outs.append(flat[off:off + ro * l].view(ro, l)[:, :co])
        off += sz
    out = []
    for i0 in range(0, n, 32):
        m = min(32, n - i0)
        P, I32, I64 = ctypes.c_void_p * m, ctypes.c_int32 * m, ctypes.c_int64 * m
        sl = slice(i0, i0 + m)
        L.call("edg_cast_batch", m, P(*[L.ptr(w) for w in ws[sl]]), P(*[L.ptr(o) for o in outs[sl]]),
               I32(*[w.shape[0] for w in ws[sl]]), I32(*[w.shape[1] for w in ws[sl]]),
               I64(*[w.stride(0) for w in ws[sl]]), I64(*lds[sl]), I32(*[int(tr) for _, tr in items[sl]]),
               L.dt(dtype), L.stream())
    return outs


def colsum(x: torch.Tensor) -> torch.Tensor:
    R, C = x.shape
    out = torch.empty((C,), dtype=torch.float32, device=x.device)
    nbytes = L.load().edg_colsum_workspace(R, C)
    ws = torch.empty(max(nbytes // 4, 1), dtype=torch.float32, device=x.device)
    L.call("edg_colsum", L.ptr(x), L.dt(x), ld(x), R, C, L.ptr(out), 0, L.ptr(ws), ws.numel() * 4, L.stream())
    return out


def trigger_gather(x: torch.Tensor, graph, anchor: torch.Tensor, lead_sigmoid: bool, want_raw: bool = True):
    B, D = graph.n_graphs, x.shape[1]
    raw = torch.empty((B, D), dtype=torch.float32, device=x.device) if want_raw else None
    act = alloc_rows(B, D, x.dtype, x.device)               # the kernel zeroes the padding columns
    L.call("edg_trigger_gather", L.ptr(x), L.dt(x), ld(x), L.ptr(graph.sent_ptr), L.ptr(anchor), B, D, L.ptr(raw),
           L.ptr(act), ld(act), int(lead_sigmoid), L.stream())
    return raw, act


def trigger_scatter_add(da: Optional[torch.Tensor], graph, anchor: torch.Tensor, dx: torch.Tensor,
                        extra: Optional[torch.Tensor] = None) -> None:
    """``dx[trigger row of b] += da[b] + extra.sum(0)[b]``; ``da`` fp32 ``[B,D]`` or None, ``extra`` fp32 ``[K,B,D]`` or None."""
    if extra is not None:
        extra = _f32c(extra)
    if da is not None:
        da = _f32c(da)
    B, D = (da.shape if da is not None else extra.shape[1:])
    L.call("edg_trigger_scatter_add", L.ptr(da), L.ptr(extra), extra.shape[0] if extra is not None else 0, B, D,
           L.ptr(graph.sent_ptr), L.ptr(anchor), L.ptr(dx), L.dt(dx), ld(dx), L.stream())


def pool_fwd(h: torch.Tensor, graph, gates: torch.Tensor, want_hmax: bool = False):
    """gates fp32 [V,B,D] -> pooled fp32 [V,B,D], arg int32 [V,B,D] (+ hmax fp32 [B,D], the plain column maximum)."""
    V, B, D = gates.shape
    pooled = torch.empty((V, B, D), dtype=torch.float32, device=h.device)
    arg = torch.empty((V, B, D), dtype=torch.int32, device=h.device)
    hmax = torch.empty((B, D), dtype=torch.float32, device=h.device) if want_hmax else None
    L.call("edg_pool_fwd", L.ptr(h), L.dt(h), ld(h), L.ptr(graph.sent_ptr), B, D, L.ptr(gates), V, L.ptr(pooled),
           L.ptr(arg), L.ptr(graph.row_sent), graph.n_rows, graph.max_len, L.ptr(hmax), L.stream())
    if want_hmax:
        return pooled, arg, hmax
    return pooled, arg


def diversity_fwd(pooled: torch.Tensor) -> torch.Tensor:
    V, B, D = pooled.shape
    xy = torch.empty((), dtype=torch.float32, device=pooled.device)
    ws = torch.empty(1024, dtype=torch.float32, device=pooled.device)
    L.call("edg_diversity_fwd", L.ptr(pooled), V, B, D, L.ptr(xy), L.ptr(ws), L.stream())
    return xy


def views_bwd(pooled, arg, gates, h, g_xy, g_pooled, dh, dgates, acc_view: int = -1, parts: int = 3) -> None:
    """``parts & 1``: add the views' gradient into ``dh``; ``parts & 2``: write ``dgates``."""
    V, B, D = pooled.shape
    L.call("edg_views_bwd_parts", L.ptr(pooled), L.ptr(arg), L.ptr(gates), L.ptr(h), L.dt(h), ld(h), V, B, D, L.ptr(g_xy),
           L.ptr(g_pooled), L.ptr(dh), ld(dh) if dh is not None else 0, L.ptr(dgates), int(acc_view), int(parts), L.stream())


def _dist_flag(dist: torch.Tensor) -> int:
    if dist.dtype == torch.int64:
        return 1
    if dist.dtype == torch.int32:
        return 0
    raise L.EdgError("dist_to_target must be int32 or int64")


def scores_kl_fwd(h, graph, gate, v, c, dist, want_units: bool = False, want_rows: bool = False):
    """``want_units``: also ``dv_unit [B,D]``, ``dc_unit [B]`` (d kl / d v, d kl / d c per unit upstream gradient);
    ``want_rows`` (with units): also ``u_unit [N]`` = d kl / d scores and ``sf_unit [B,D]`` = sum_t u_t h_t, the
    inputs of :func:`head_du`."""
    B, D = gate.shape
    N = h.shape[0]
    scores = torch.empty((N,), dtype=torch.float32, device=h.device)
    kl_b = torch.empty((B,), dtype=torch.float32, device=h.device)
    dvu = torch.empty((B, D), dtype=torch.float32, device=h.device) if want_units else None
    dcu = torch.empty((B,), dtype=torch.float32, device=h.device) if want_units else None
    uu = torch.empty((N,), dtype=torch.float32, device=h.device) if want_units and want_rows else None
    sfu = torch.empty((B, D), dtype=torch.float32, device=h.device) if want_units and want_rows else None
    L.call("edg_scores_kl_fwd", L.ptr(h), L.dt(h), ld(h), L.ptr(graph.sent_ptr), B, D, L.ptr(gate), L.ptr(v),
           L.ptr(c), L.ptr(dist), _dist_flag(dist), L.ptr(scores), L.ptr(kl_b), L.ptr(dvu), L.ptr(dcu), L.ptr(uu), L.ptr(sfu),
           L.ptr(graph.row_sent), graph.n_rows, graph.max_len, L.stream())
    kl = torch.empty((), dtype=torch.float32, device=h.device)
    L.call("edg_sum_scaled", L.ptr(kl_b), B, 1.0 / B, L.ptr(kl), L.stream())
    if want_units and want_rows:
        return scores, kl_b, kl, dvu, dcu, uu, sfu
    if want_units:
        return scores, kl_b, kl, dvu, dcu
    return scores, kl_b, kl


def fc_head_fwd(logits: torch.Tensor, fc_w: torch.Tensor, fc_b: torch.Tensor, a: torch.Tensor):
    """``[v | va] = logits @ fc_w``, ``c = a . va + logits . fc_b`` (fp32): v [B,D], c [B]."""
    B, C = logits.shape
    D = a.shape[1]
    v = torch.empty((B, D), dtype=torch.float32, device=a.device)
    c = torch.empty((B,), dtype=torch.float32, device=a.device)
    L.call("edg_fc_head_fwd", L.ptr(logits), ld(logits), L.ptr(fc_w), ld(fc_w), L.ptr(fc_b), L.ptr(a), ld(a), B, D, C,
           L.ptr(v), L.ptr(c), L.stream())
    return v, c


def fc_head_bwd(logits, fc_w, fc_b, a, dv, dc, scale: Optional[torch.Tensor] = None, parts: int = 3):
    """Backward of :func:`fc_head_fwd` -> d_logits [B,C], d_a [B,D] (``parts & 1``), d_fc_w [C,2D], d_fc_b [C]
    (``parts & 2``); ``dv``/``dc`` are multiplied by the device scalar ``scale`` when given."""
    B, C = logits.shape
    D = a.shape[1]
    dev = a.device
    d_lg = torch.empty((B, C), dtype=torch.float32, device=dev) if parts & 1 else None
    d_a = torch.empty((B, D), dtype=torch.float32, device=dev) if parts & 1 else None
    d_w = torch.empty((C, 2 * D), dtype=torch.float32, device=dev) if parts & 2 else None
    d_b = torch.empty((C,), dtype=torch.float32, device=dev) if parts & 2 else None
    nbytes = L.load().edg_fc_head_bwd_workspace(B, D, C)
    ws = torch.empty((nbytes + 3) // 4, dtype=torch.float32, device=dev)
    L.call("edg_fc_head_bwd", L.ptr(logits), ld(logits), L.ptr(fc_w), ld(fc_w), L.ptr(fc_b), L.ptr(a), ld(a),
           L.ptr(dv), L.ptr(dc), L.ptr(scale), B, D, C, int(parts), L.ptr(d_lg), C, L.ptr(d_a), L.ptr(d_w), 2 * D,
           L.ptr(d_b), L.ptr(ws), ws.numel() * 4, L.stream())
    return d_lg, d_a, d_w, d_b


DENSE_HEAD_MAX_CLASSES = 64


def dense_head_fwd(a: torch.Tensor, p: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor]) -> torch.Tensor:
    """``edg_dense_head_fwd``: ``cat([a, p], 1) @ w.T + bias`` with ``a, p`` fp32 ``[B, D]``, ``w`` fp32 ``[C, 2D]``."""
    a, p, w = _f32c(a), _f32c(p), _f32c(w)
    B, D = a.shape
    C = w.shape[0]
    assert p.shape == (B, D) and w.shape[1] == 2 * D
    bias = _f32c(bias) if bias is not None else None
    logits = torch.empty((B, C), dtype=torch.float32, device=a.device)
    L.call("edg_dense_head_fwd", L.ptr(a), ld(a), L.ptr(p), ld(p), L.ptr(w), ld(w), L.ptr(bias), B, D, C,
           L.ptr(logits), C, L.stream())
    return logits


def dense_head_bwd(g: torch.Tensor, a: torch.Tensor, p: torch.Tensor, w: torch.Tensor, parts: int = 3,
                   g2: Optional[torch.Tensor] = None, da_add: Optional[torch.Tensor] = None,
                   dp_add: Optional[torch.Tensor] = None):
    """``edg_dense_head_bwd`` -> ``(da [B,D], dp [B,D])`` (``parts & 1``), ``(dW [C,2D], dbias [C])`` (``parts & 2``)
    from ``d logits = g (+ g2) [B,C]``; ``da_add`` / ``dp_add`` (fp32 ``[B,D]``) are added to ``da`` / ``dp``."""
    g, a, p, w = _f32c(g), _f32c(a), _f32c(p), _f32c(w)
    g2 = _f32c(g2) if g2 is not None else None
    da_add = _f32c(da_add) if da_add is not None else None
    dp_add = _f32c(dp_add) if dp_add is not None else None
    B, D = a.shape
    C = w.shape[0]
    dev = a.device
    da = torch.empty((B, D), dtype=torch.float32, device=dev) if parts & 1 else None
    dp = torch.empty((B, D), dtype=torch.float32, device=dev) if parts & 1 else None
    dW = torch.empty((C, 2 * D), dtype=torch.float32, device=dev) if parts & 2 else None
    db = torch.empty((C,), dtype=torch.float32, device=dev) if parts & 2 else None
    nbytes = L.load().edg_dense_head_bwd_workspace(B, D, C)
    ws = torch.empty((nbytes + 3) // 4, dtype=torch.float32, device=dev)
    L.call("edg_dense_head_bwd", L.ptr(g), ld(g), L.ptr(a), ld(a), L.ptr(p), ld(p), L.ptr(w), ld(w), B, D, C, int(parts),
           L.ptr(g2), ld(g2) if g2 is not None else 0, L.ptr(da_add), L.ptr(dp_add),
           L.ptr(da), L.ptr(dp), L.ptr(dW), 2 * D, L.ptr(db), L.ptr(ws), ws.numel() * 4, L.stream())
    return da, dp, dW, db


def block_head_fwd(a, a_fc, p, g, w, bias, fc_w, fc_b):
    """``edg_block_head_fwd``: ``pooled = g * p`` (``p`` itself when ``g`` is None), ``logits = cat([a, pooled]) @ w.T
    + bias``, and the scores' operands ``v = logits @ fc_w[:, :D]``, ``c = logits . (fc_w[:, D:] a_fc + fc_b)`` in one
    launch.  All fp32 ``[B, D]`` rows.  Returns ``(pooled, logits [B,C], v [B,D], c [B])``."""
    a, a_fc, p, w, fc_w, fc_b = (_f32c(t) for t in (a, a_fc, p, w, fc_w, fc_b))
    g = _f32c(g) if g is not None else None
    bias = _f32c(bias) if bias is not None else None
    B, D = a.shape
    C = w.shape[0]
    assert p.shape == (B, D) and a_fc.shape == (B, D) and w.shape[1] == 2 * D and fc_w.shape == (C, 2 * D)
    dev = a.device
    pooled = torch.empty((B, D), dtype=torch.float32, device=dev) if g is not None else p
    logits = torch.empty((B, C), dtype=torch.float32, device=dev)
    v = torch.empty((B, D), dtype=torch.float32, device=dev)
    c = torch.empty((B,), dtype=torch.float32, device=dev)
    L.call("edg_block_head_fwd", L.ptr(a), ld(a), L.ptr(a_fc), ld(a_fc), L.ptr(p), ld(p), L.ptr(g),
           ld(g) if g is not None else 0, L.ptr(w), ld(w), L.ptr(bias), L.ptr(fc_w), ld(fc_w), L.ptr(fc_b), B, D, C,
           L.ptr(pooled) if g is not None else None, L.ptr(logits), L.ptr(v), L.ptr(c), L.stream())
    return pooled, logits, v, c


def block_head_bwd(logits, a, a_fc, fc_sigmoid: bool, w, fc_w, fc_b, dv=None, dc=None, scale=None, g_logits=None,
                   g_pooled=None):
    """``edg_block_head_bwd`` -> ``(d logits [B,C], d a [B,D], d pooled [B,D])`` of :func:`block_head_fwd`, with the
    scores' ``dv`` / ``dc`` (times the device scalar ``scale``; both None when the scores carry no gradient) and the
    direct gradients ``g_logits`` / ``g_pooled`` (each optional) flowing in."""
    logits, a, a_fc, w, fc_w, fc_b = (_f32c(t) for t in (logits, a, a_fc, w, fc_w, fc_b))
    dv, dc, scale, g_logits, g_pooled = (_f32c(t) if t is not None else None for t in (dv, dc, scale, g_logits, g_pooled))
    B, D = a.shape
    C = w.shape[0]
    dev = a.device
    dlg = torch.empty((B, C), dtype=torch.float32, device=dev)
    da = torch.empty((B, D), dtype=torch.float32, device=dev)
    dp = torch.empty((B, D), dtype=torch.float32, device=dev)
    L.call("edg_block_head_bwd", L.ptr(logits), L.ptr(a), ld(a), L.ptr(a_fc), ld(a_fc), int(bool(fc_sigmoid)), L.ptr(w),
           ld(w), L.ptr(fc_w), ld(fc_w), L.ptr(fc_b), L.ptr(dv), L.ptr(dc), L.ptr(scale), L.ptr(g_logits),
           L.ptr(g_pooled), B, D, C, L.ptr(dlg), L.ptr(da), L.ptr(dp), L.stream())
    return dlg, da, dp


def block_head_wgrad(logits, dlg, a, a_fc, pooled, dv=None, dc=None, scale=None, want_bias: bool = True):
    """``edg_block_head_wgrad`` -> ``(dW [C,2D], dbias [C], d fc_w [C,2D], d fc_b [C])``: the head's parameter gradients
    when ``dlg`` is given (``dbias`` None unless ``want_bias``), the fc's when ``dv`` / ``dc`` are (else None)."""
    logits, a, a_fc, pooled = (_f32c(t) for t in (logits, a, a_fc, pooled))
    dlg, dv, dc, scale = (_f32c(t) if t is not None else None for t in (dlg, dv, dc, scale))
    B, D = a.shape
    C = logits.shape[1]
    dev = a.device
    new = lambda *s: torch.empty(s, dtype=torch.float32, device=dev)
    dW, dbias = (new(C, 2 * D), new(C) if want_bias else None) if dlg is not None else (None, None)
    d_fw, d_fb = (new(C, 2 * D), new(C)) if dv is not None else (None, None)
    nbytes = L.load().edg_block_head_wgrad_workspace(B, D, C)
    ws = torch.empty((nbytes + 3) // 4, dtype=torch.float32, device=dev)
    L.call("edg_block_head_wgrad", L.ptr(logits), L.ptr(dlg), L.ptr(a), ld(a), L.ptr(a_fc), ld(a_fc), L.ptr(pooled),
           ld(pooled), L.ptr(dv), L.ptr(dc), L.ptr(scale), B, D, C, L.ptr(dW), L.ptr(dbias), L.ptr(d_fw), L.ptr(d_fb),
           L.ptr(ws), ws.numel() * 4, L.stream())
    return dW, dbias, d_fw, d_fb


def cross_entropy_fwd(logits: torch.Tensor, target: torch.Tensor, ignore_index: int = -100):
    """``edg_cross_entropy_fwd`` -> ``(out fp32 [2] = {mean loss, counted rows}, bad int32 [1])``."""
    B, C = logits.shape
    out = torch.empty((2,), dtype=torch.float32, device=logits.device)
    nbytes = L.load().edg_cross_entropy_workspace(B)
    # one zeroed allocation: [bad flag | per-block partial sums | ticket counter]
    buf = torch.zeros((1 + (nbytes + 3) // 4,), dtype=torch.int32, device=logits.device)
    bad, ws = buf[:1], buf[1:]
    L.call("edg_cross_entropy_fwd", L.ptr(logits), ld(logits), L.ptr(target), B, C, int(ignore_index), L.ptr(out),
           L.ptr(bad), L.ptr(ws), ws.numel() * 4, L.stream())
    return out, bad


def cross_entropy_bwd(logits: torch.Tensor, target: torch.Tensor, gscale: Optional[torch.Tensor], fwd_out: torch.Tensor,
                      ignore_index: int = -100) -> torch.Tensor:
    B, C = logits.shape
    dlg = torch.empty((B, C), dtype=torch.float32, device=logits.device)
    L.call("edg_cross_entropy_bwd", L.ptr(logits), ld(logits), L.ptr(target), B, C, int(ignore_index), L.ptr(gscale),
           L.ptr(fwd_out), L.ptr(dlg), C, L.stream())
    return dlg


def head_bwd(h, graph, gate, v, dist, scores, kl_b, g_kl, g_scores, g_pooled, arg, g_xout, want_dh: bool,
             want_dv: bool, dgate_out: Optional[torch.Tensor] = None):
    B, D = gate.shape
    N = h.shape[0]
    dh = alloc_rows(N, D, h.dtype, h.device) if want_dh else None
    dgate = (dgate_out if dgate_out is not None else torch.empty((B, D), dtype=torch.float32, device=h.device)) \
        if want_dh else None
    dv = torch.empty((B, D), dtype=torch.float32, device=h.device) if want_dv else None
    dc = torch.empty((B,), dtype=torch.float32, device=h.device) if want_dv else None
    L.call("edg_head_bwd", L.ptr(h), L.dt(h), ld(h), L.ptr(graph.sent_ptr), B, D, L.ptr(gate), L.ptr(v),
           L.ptr(dist), _dist_flag(dist) if dist is not None else 0, L.ptr(scores), L.ptr(kl_b), L.ptr(g_kl),
           L.ptr(g_scores), L.ptr(g_pooled), L.ptr(arg), L.ptr(g_xout), ld(g_xout) if g_xout is not None else 0,
           L.ptr(dh), ld(dh) if dh is not None else 0, L.ptr(dgate), L.ptr(dv), L.ptr(dc), graph.max_len,
           L.ptr(graph.row_sent), graph.n_rows, L.stream())
    return dh, dgate, dv, dc


def gate_rows(h, graph, gate, out_dtype, act: int = L.ACT_NONE):
    """``act(gate[b] * h[t])`` per row (act = none or sigmoid); padding columns zero."""
    B, D = gate.shape
    out = alloc_rows(h.shape[0], D, out_dtype, h.device, zero=True)
    L.call("edg_gate_rows_act", L.ptr(h), L.dt(h), ld(h), L.ptr(graph.sent_ptr), B, D, L.ptr(gate), L.ptr(out),
           L.dt(out), ld(out), int(act), L.stream())
    return out


def sigmoid_bwd(y: torch.Tensor, dy: torch.Tensor, out_dtype: torch.dtype, out: Optional[torch.Tensor] = None,
                accumulate: bool = False) -> torch.Tensor:
    """dz (+)= dy * y * (1 - y); the kernel also zeroes dz's padding columns."""
    R, C = y.shape
    dz = out if out is not None else alloc_rows(R, C, out_dtype, y.device)
    L.call("edg_sigmoid_bwd", L.ptr(y), L.dt(y), ld(y), L.ptr(dy), L.dt(dy), ld(dy), R, C, L.ptr(dz), L.dt(dz),
           ld(dz), int(accumulate), L.stream())
    return dz


def dropout_rows(x: torch.Tensor, seed: torch.Tensor, stream_id: int, p: float, out: Optional[torch.Tensor] = None,
                 accumulate: bool = False) -> torch.Tensor:
    """``out (+)= x * keep / (1 - p)`` with the counter-based per-(row, column) mask of ``edg_dropout_rows``
    (``seed`` = device int64 scalar)."""
    N, D = x.shape
    if out is None:
        out = alloc_rows(N, D, x.dtype, x.device)
    L.call("edg_dropout_rows", L.ptr(x), L.dt(x), ld(x), L.ptr(out), ld(out), N, D, L.ptr(seed), int(stream_id), float(p),
           int(accumulate), L.stream())
    return out


# ---------------------------------------------------------------------------
# (sentence, trigger) pairs over sentence rows (graph.TriggerPairs; include/edgcn.h "Trigger pairs")
class PairRows:
    """The pairs seen as B = P 'sentences' starting at ``pair_start``: what ``edg_trigger_gather`` reads (``sent_ptr[b]``
    only), so the per-pair trigger rows of the sentence rows come from the existing gather."""
    __slots__ = ("sent_ptr", "n_graphs")

    def __init__(self, pairs):
        self.sent_ptr, self.n_graphs = pairs.pair_start, pairs.n_pairs


def scores_kl_pairs_fwd(h, graph, pairs, gate, v, c, dist, want_units: bool = True):
    """``edg_scores_kl_pairs_fwd`` -> ``(scores [n_pair_rows], kl_b [P], kl, dv_unit [P,D], dc_unit [P])`` (units None
    without ``want_units``); ``kl`` is the mean over the P pairs."""
    P, D = gate.shape
    dev = h.device
    R = pairs.n_pair_rows
    scores = torch.empty((max(R, 1),), dtype=torch.float32, device=dev)[:R]
    kl_b = torch.empty((P,), dtype=torch.float32, device=dev)
    dvu = torch.empty((P, D), dtype=torch.float32, device=dev) if want_units else None
    dcu = torch.empty((P,), dtype=torch.float32, device=dev) if want_units else None
    L.call("edg_scores_kl_pairs_fwd", L.ptr(h), L.dt(h), ld(h), L.ptr(graph.sent_ptr), L.ptr(pairs.pair_sent),
           L.ptr(pairs.pair_row_ptr), P, D, L.ptr(gate), L.ptr(v), L.ptr(c), L.ptr(dist), _dist_flag(dist), L.ptr(scores),
           L.ptr(kl_b), L.ptr(dvu), L.ptr(dcu), None, None, L.stream())
    kl = torch.empty((), dtype=torch.float32, device=dev)
    L.call("edg_sum_scaled", L.ptr(kl_b), P, 1.0 / max(P, 1), L.ptr(kl), L.stream())
    return scores, kl_b, kl, dvu, dcu


def head_bwd_pairs(h, graph, pairs, gate, v, dist, scores, kl_b, g_kl, g_scores, g_pooled, arg, want_dh: bool,
                   dgate_out: Optional[torch.Tensor] = None):
    """``edg_head_bwd_pairs``.  ``want_dh``: the full pass -> ``(dh [N,D] compute dtype, dgate [P,D], None, None)``;
    otherwise the first pass -> ``(None, None, dv [P,D], dc [P])``.  ``arg`` int32 [S,D] = the sentences' arg-max rows."""
    P, D = gate.shape
    N = h.shape[0]
    dev = h.device
    dh = alloc_rows(N, D, h.dtype, dev) if want_dh else None
    dgate = (dgate_out if dgate_out is not None else torch.empty((P, D), dtype=torch.float32, device=dev)) \
        if want_dh else None
    dv = None if want_dh else torch.empty((P, D), dtype=torch.float32, device=dev)
    dc = None if want_dh else torch.empty((P,), dtype=torch.float32, device=dev)
    ds_ws = torch.empty((max(pairs.n_pair_rows, 1),), dtype=torch.float32, device=dev)
    if want_dh and graph.row_sent is None:
        raise L.EdgError("the pairs head backward needs graph.row_sent (build_graph / graph_from_dense set it)")
    L.call("edg_head_bwd_pairs", L.ptr(h), L.dt(h), ld(h), L.ptr(graph.sent_ptr), graph.n_graphs,
           L.ptr(graph.row_sent) if N > 0 else None, N, L.ptr(pairs.pair_ptr),
           L.ptr(pairs.pair_sent), L.ptr(pairs.pair_row_ptr), P, D, L.ptr(gate), L.ptr(v), L.ptr(dist),
           _dist_flag(dist) if dist is not None else 0, L.ptr(scores), L.ptr(kl_b), L.ptr(g_kl), L.ptr(g_scores),
           L.ptr(g_pooled), L.ptr(arg), L.ptr(dh), ld(dh) if dh is not None else 0, L.ptr(dgate), L.ptr(dv), L.ptr(dc),
           L.ptr(ds_ws), L.stream())
    return dh, dgate, dv, dc


def views_bwd_hmax_pairs(hmax: torch.Tensor, gates: torch.Tensor, g_xy, dgates: torch.Tensor, pairs,
                         acc_view: int = -1) -> torch.Tensor:
    """``edg_views_bwd_hmax_pairs``: writes ``dgates [V,P,D]`` and returns ``patch_val fp32 [S,D]`` (what the arg-max
    rows of the sentences' d h_1 receive)."""
    V, P, D = gates.shape
    S = hmax.shape[0]
    patch_val = torch.empty((S, D), dtype=torch.float32, device=hmax.device)
    L.call("edg_views_bwd_hmax_pairs", L.ptr(hmax), L.ptr(gates), L.ptr(g_xy), V, S, L.ptr(pairs.pair_ptr), P, D,
           L.ptr(patch_val), D, L.ptr(dgates), int(acc_view), L.stream())
    return patch_val


def pool_drop_pairs(h, graph, pairs, gates: torch.Tensor, seed: torch.Tensor, stream0: int, p: float):
    """``edg_pool_drop_pairs``: the gated max-pool of every pair's masked rows, view v under dropout stream
    ``stream0 + v`` -> ``(pooled fp32 [V,P,D], arg int32 [V,P,D] (global sentence rows), mmax fp32 [V,P,D])``."""
    V, P, D = gates.shape
    dev = h.device
    pooled = torch.empty((V, P, D), dtype=torch.float32, device=dev)
    arg = torch.empty((V, P, D), dtype=torch.int32, device=dev)
    mmax = torch.empty((V, P, D), dtype=torch.float32, device=dev)
    L.call("edg_pool_drop_pairs", L.ptr(h), L.dt(h), ld(h), L.ptr(graph.sent_ptr), L.ptr(pairs.pair_sent),
           L.ptr(pairs.pair_row_ptr), P, D, L.ptr(gates.contiguous()), V, L.ptr(seed), int(stream0), float(p),
           L.ptr(pooled), L.ptr(arg), L.ptr(mmax), L.stream())
    return pooled, arg, mmax


def scores_kl_drop_pairs_fwd(h, graph, pairs, gate, v, c, dist, seed: torch.Tensor, stream_id: int, p: float):
    """:func:`scores_kl_pairs_fwd` on the pairs' masked rows of dropout stream ``stream_id``."""
    P, D = gate.shape
    dev = h.device
    R = pairs.n_pair_rows
    scores = torch.empty((max(R, 1),), dtype=torch.float32, device=dev)[:R]
    kl_b = torch.empty((P,), dtype=torch.float32, device=dev)
    dvu = torch.empty((P, D), dtype=torch.float32, device=dev)
    dcu = torch.empty((P,), dtype=torch.float32, device=dev)
    L.call("edg_scores_kl_drop_pairs_fwd", L.ptr(h), L.dt(h), ld(h), L.ptr(graph.sent_ptr), L.ptr(pairs.pair_sent),
           L.ptr(pairs.pair_row_ptr), P, D, L.ptr(gate), L.ptr(v), L.ptr(c), L.ptr(dist), _dist_flag(dist), L.ptr(scores),
           L.ptr(kl_b), L.ptr(dvu), L.ptr(dcu), None, None, L.ptr(seed), int(stream_id), float(p), L.stream())
    kl = torch.empty((), dtype=torch.float32, device=dev)
    L.call("edg_sum_scaled", L.ptr(kl_b), P, 1.0 / max(P, 1), L.ptr(kl), L.stream())
    return scores, kl_b, kl, dvu, dcu


def head_bwd_drop_pairs(h, graph, pairs, gate, v, dist, scores, kl_b, g_kl, g_scores, g_pooled, arg, mmax,
                        seed: torch.Tensor, stream_id: int, p: float, want_dh: bool,
                        dgate_out: Optional[torch.Tensor] = None):
    """:func:`head_bwd_pairs` on the pairs' masked rows of dropout stream ``stream_id``; ``arg`` int32 / ``mmax`` fp32
    ``[P,D]`` are the final pool's per-pair arg-max rows and masked maxima (:func:`pool_drop_pairs`)."""
    P, D = gate.shape
    N = h.shape[0]
    dev = h.device
    dh = alloc_rows(N, D, h.dtype, dev) if want_dh else None
    dgate = (dgate_out if dgate_out is not None else torch.empty((P, D), dtype=torch.float32, device=dev)) \
        if want_dh else None
    dv = None if want_dh else torch.empty((P, D), dtype=torch.float32, device=dev)
    dc = None if want_dh else torch.empty((P,), dtype=torch.float32, device=dev)
    ds_ws = torch.empty((max(pairs.n_pair_rows, 1),), dtype=torch.float32, device=dev)
    if want_dh and graph.row_sent is None:
        raise L.EdgError("the pairs head backward needs graph.row_sent (build_graph / graph_from_dense set it)")
    L.call("edg_head_bwd_drop_pairs", L.ptr(h), L.dt(h), ld(h), L.ptr(graph.sent_ptr), graph.n_graphs,
           L.ptr(graph.row_sent) if N > 0 else None, N, L.ptr(pairs.pair_ptr),
           L.ptr(pairs.pair_sent), L.ptr(pairs.pair_row_ptr), P, D, L.ptr(gate), L.ptr(v), L.ptr(dist),
           _dist_flag(dist) if dist is not None else 0, L.ptr(scores), L.ptr(kl_b), L.ptr(g_kl), L.ptr(g_scores),
           L.ptr(g_pooled), L.ptr(arg), L.ptr(mmax), L.ptr(dh), ld(dh) if dh is not None else 0, L.ptr(dgate), L.ptr(dv),
           L.ptr(dc), L.ptr(ds_ws), L.ptr(seed), int(stream_id), float(p), L.stream())
    return dh, dgate, dv, dc


def views_bwd_drop_pairs(pooled, mmax, arg, gates, g_xy, graph, pairs, seed: torch.Tensor, p: float,
                         dh: Optional[torch.Tensor] = None, dgates: Optional[torch.Tensor] = None,
                         acc_view: int = -1) -> None:
    """``edg_views_bwd_drop_pairs`` for the views of :func:`pool_drop_pairs` (streams 0..V-1): writes ``dgates
    [V,P,D]`` (``acc_view`` accumulates) and / or adds the views' share of d h_1 into ``dh``."""
    V, P, D = pooled.shape
    N = graph.n_rows
    if dh is not None and graph.row_sent is None:
        raise L.EdgError("the pairs views backward needs graph.row_sent (build_graph / graph_from_dense set it)")
    L.call("edg_views_bwd_drop_pairs", L.ptr(pooled), L.ptr(mmax), L.ptr(arg), L.ptr(gates), L.ptr(g_xy), V,
           L.ptr(graph.sent_ptr), L.ptr(graph.row_sent) if (dh is not None and N > 0) else None, N, L.ptr(pairs.pair_ptr),
           L.ptr(pairs.pair_row_ptr), P, D, L.ptr(seed), float(p), L.ptr(dh), L.dt(dh) if dh is not None else 0,
           ld(dh) if dh is not None else 0, L.ptr(dgates), int(acc_view), L.stream())


def trigger_scatter_add_pairs(da: Optional[torch.Tensor], pairs, anchor: torch.Tensor, dx: torch.Tensor,
                              extra: Optional[torch.Tensor] = None) -> None:
    """``dx[pair_start[p] + anchor[p]] += da[p] + extra.sum(0)[p]`` in pair order per sentence (anchors may repeat)."""
    if extra is not None:
        extra = _f32c(extra)
    if da is not None:
        da = _f32c(da)
    P, D = (da.shape if da is not None else extra.shape[1:])
    L.call("edg_trigger_scatter_add_pairs", L.ptr(da), L.ptr(extra), extra.shape[0] if extra is not None else 0,
           pairs.n_sentences, L.ptr(pairs.pair_ptr), P, D, L.ptr(pairs.pair_start), L.ptr(anchor), L.ptr(dx), L.dt(dx),
           ld(dx), L.stream())
