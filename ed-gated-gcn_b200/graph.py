"""Dependency-tree adjacency and distance-to-trigger on the GPU.

Replaces, for the training-time path, the dense ``eye(100) + symmetric edges``
matrix of ``graph.py:66-75`` and the recursive ``get_dist_to_target`` of
``data_utils.py:302-323`` with integer kernels over a packed CSR of many
sentences (bit-exact against the reference on trees / forests).
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Optional

import torch

from . import _lib as L


@dataclass
class DepGraph:
    """Packed CSR of B sentences.  Row ``i`` of sentence ``b`` is global row
    ``sent_ptr[b] + i``; ``col[row_ptr[r]:row_ptr[r+1]]`` lists the global rows of
    self + parent + children in ascending order (the non-zeros of graph.py:66-75)."""
    sent_ptr: torch.Tensor        # int32 [B+1]
    row_ptr: torch.Tensor         # int32 [N+1]
    col: torch.Tensor             # int32 [>= nnz]
    row_sent: Optional[torch.Tensor]   # int32 [N]
    n_graphs: int
    n_rows: int
    max_len: int
    padded_T: Optional[int] = None     # set when built from a dense [B,T,T] batch
    max_sent_nnz: Optional[int] = None  # largest CSR entry count of one sentence (None: a tree, 3n - 2)

    @property
    def device(self):
        return self.row_ptr.device

    def tile_plan(self, max_rows: int):
        """Sentence-aligned row tiles for the fused layer kernel (``edg_gcn_layer``): ``(tile_info int32
        [B+1, 8], n_tiles int32 [1])``, built by one small kernel on first use and cached per ``max_rows``.
        ``None`` when a sentence cannot fit a tile (the caller then runs the unfused kernels)."""
        if self.max_len > max_rows or self.n_graphs == 0:
            return None
        if (self.max_sent_nnz if self.max_sent_nnz is not None else 3 * self.max_len) > 512:
            return None
        plans = self.__dict__.setdefault("_plans", {})
        plan = plans.get(max_rows)
        if plan is None:
            dev = self.device
            info = torch.empty((self.n_graphs + 1, 8), dtype=torch.int32, device=dev)
            n_tiles = torch.empty(1, dtype=torch.int32, device=dev)
            with torch.cuda.device(dev):
                L.call("edg_tile_plan", L.ptr(self.sent_ptr), L.ptr(self.row_ptr), self.n_graphs, int(max_rows),
                       L.ptr(info), L.ptr(n_tiles), L.stream())
            plan = plans[max_rows] = (info, n_tiles)
        return plan


@dataclass
class TriggerPairs:
    """(sentence, candidate trigger) pairs over the sentences of a ``DepGraph``, grouped by sentence: the pairs of
    sentence ``s`` are ``pair_ptr[s] .. pair_ptr[s+1] - 1`` (a sentence may have none; pairs may share an anchor).
    Per-pair row data (distances, scores) uses the per-pair packed layout: pair ``p``'s copy of its sentence's rows
    starts at ``pair_row_ptr[p]``.  All tensors live on the graph's device.  Built by :func:`pairs_from_ptr`."""
    pair_ptr: torch.Tensor        # int32 [S+1]
    pair_sent: torch.Tensor       # int32 [P]   sentence of every pair
    pair_start: torch.Tensor      # int32 [P]   = sent_ptr[pair_sent]: first packed row of the pair's sentence
    anchor: torch.Tensor          # int32 [P]   sentence-local trigger index
    pair_row_ptr: torch.Tensor    # int32 [P+1] offsets of the pairs' copies of their sentences
    n_pairs: int
    n_sentences: int
    n_pair_rows: int

    @property
    def device(self):
        return self.pair_ptr.device


def pairs_from_ptr(graph: DepGraph, pair_ptr: torch.Tensor, anchor: torch.Tensor,
                   n_pair_rows: Optional[int] = None) -> TriggerPairs:
    """``pair_ptr`` int ``[S+1]`` (S = ``graph.n_graphs``; monotone, ``pair_ptr[0] = 0``, ``pair_ptr[S] = P``) and the
    sentence-local ``anchor`` int ``[P]`` of every pair -> :class:`TriggerPairs`, built with torch ops on the graph's
    device.

    ``n_pair_rows`` (the sum of the pairs' sentence lengths, ``PackedBatch.n_pair_rows``) may be passed as the caller
    knows it: the build then makes no device->host read and can be captured in a CUDA graph, like
    ``build_graph(max_len=, max_sent_nnz=)``; device-side values of ``pair_ptr`` / ``anchor`` are then not checked
    (host tensors still are).  Without it one small read returns ``n_pair_rows`` together with the checks: ``pair_ptr``
    monotone from 0 to P, and every anchor inside its sentence."""
    dev = graph.device
    S = graph.n_graphs
    if pair_ptr.dim() != 1 or pair_ptr.numel() != S + 1:
        raise L.EdgError(f"pair_ptr must be int [S+1] = [{S + 1}], got {tuple(pair_ptr.shape)}")
    if anchor.dim() != 1:
        raise L.EdgError(f"anchor must be int [P], got {tuple(anchor.shape)}")
    P = anchor.numel()
    if not pair_ptr.is_cuda:                 # host-side checks cost no device read
        pp = pair_ptr.to(torch.int64)
        if int(pp[0]) != 0 or int(pp[-1]) != P or bool((pp[1:] < pp[:-1]).any()):
            raise L.EdgError(f"pair_ptr must rise monotonically from 0 to P = {P}")
    pair_ptr = _i32(pair_ptr, dev)
    anchor = _i32(anchor, dev)
    sp = graph.sent_ptr
    lens = sp[1:] - sp[:-1]
    # sentence of pair p = number of sentences whose pairs end at or before p (empty ranges included); no host read
    idx = torch.arange(P, dtype=torch.int32, device=dev)
    pair_sent = torch.searchsorted(pair_ptr[1:], idx, right=True, out_int32=True).clamp_(max=max(S - 1, 0))
    if S == 0:
        pair_sent = pair_sent[:0]
    pair_start = sp[:-1][pair_sent.long()] if P else pair_sent.clone()
    plen = lens[pair_sent.long()] if P else pair_sent.clone()
    pair_row_ptr = torch.zeros(P + 1, dtype=torch.int32, device=dev)
    if P:
        pair_row_ptr[1:] = torch.cumsum(plen, 0, dtype=torch.int32)
    if n_pair_rows is None:
        bad_ptr = (pair_ptr[0] != 0) | (pair_ptr[-1] != P) | (pair_ptr[1:] < pair_ptr[:-1]).any()
        bad_anchor = ((anchor < 0) | (anchor >= plen)).any() if P else torch.zeros((), dtype=torch.bool, device=dev)
        host = torch.stack([pair_row_ptr[-1].long(), bad_ptr.long(), bad_anchor.long()]).cpu()   # one small read
        n_pair_rows, bp, ba = (int(v) for v in host)
        if bp:
            raise L.EdgError(f"pair_ptr must rise monotonically from 0 to P = {P}")
        if ba:
            raise L.EdgError("a pair's anchor lies outside its sentence")
    return TriggerPairs(pair_ptr, pair_sent.contiguous(), pair_start.contiguous(), anchor, pair_row_ptr, P, S,
                        int(n_pair_rows))


def _i32(t: torch.Tensor, device) -> torch.Tensor:
    return t.to(device=device, dtype=torch.int32).contiguous()


def build_graph(heads: torch.Tensor, sent_ptr: torch.Tensor, max_len: Optional[int] = None,
                device: Optional[torch.device] = None, extra_edges: Optional[torch.Tensor] = None,
                edge_ptr: Optional[torch.Tensor] = None, max_sent_nnz: Optional[int] = None) -> DepGraph:
    """heads int [N] (sentence-local head index, -1 = root), sent_ptr int [B+1].

    The packed counterpart of ``gen_graph`` (graph.py:62-75).  ``max_len`` (longest
    sentence) may be passed to avoid one device->host read.

    Graphs that are not forests (enhanced dependencies, graph.py:63-64) come as the forest of ``heads`` plus
    ``extra_edges`` int [E, 2] of sentence-local undirected pairs, sentence b owning pairs ``edge_ptr[b]`` ..
    ``edge_ptr[b+1] - 1`` (``wire.split_adjacency`` / ``collate_packed`` produce both).  Pairs follow set semantics:
    duplicates, reversed pairs, pairs that repeat a head edge and self pairs change nothing; pairs with an endpoint
    outside the sentence are dropped.  The graph then carries ``max_sent_nnz``, the largest CSR entry count of one
    sentence (it decides whether the fused layer kernels can take the batch).  ``max_sent_nnz`` may be passed as an
    upper bound the caller guarantees, like ``max_len`` (``PackedBatch.max_sent_nnz`` is exact); the kernels trap on a
    sentence above it.  With both ``max_len`` and ``max_sent_nnz`` given the build makes no device->host read and can
    be captured in a CUDA graph.  Otherwise a missing ``max_sent_nnz`` is read back after the build (one 4-byte copy),
    and a missing ``max_len`` is computed from ``sent_ptr`` before it (a read only when ``sent_ptr`` is on the GPU).
    Without ``extra_edges``, ``edge_ptr`` and ``max_sent_nnz`` are ignored."""
    device = torch.device(device) if device is not None else heads.device
    if device.type != "cuda":
        raise L.EdgError("build_graph needs a CUDA device (there is no CPU path)")
    if extra_edges is not None:
        return _build_graph_edges(heads, sent_ptr, max_len, device, extra_edges, edge_ptr, max_sent_nnz)
    heads = _i32(heads, device)
    sent_ptr = _i32(sent_ptr, device)
    B = sent_ptr.numel() - 1
    N = heads.numel()
    if max_len is None:
        max_len = int((sent_ptr[1:] - sent_ptr[:-1]).max().item()) if B > 0 else 0
    row_ptr = torch.empty(N + 1, dtype=torch.int32, device=device)
    col = torch.empty(max(3 * N, 1), dtype=torch.int32, device=device)
    row_sent = torch.empty(max(N, 1), dtype=torch.int32, device=device)
    ws = torch.empty(B + 2, dtype=torch.int32, device=device)
    with torch.cuda.device(device):
        L.call("edg_csr_from_heads", L.ptr(heads), L.ptr(sent_ptr), B, N, max_len, L.ptr(row_ptr), L.ptr(col),
               L.ptr(row_sent), L.ptr(ws), L.stream())
    return DepGraph(sent_ptr, row_ptr, col, row_sent[:N], B, N, max_len)


def _build_graph_edges(heads, sent_ptr, max_len, device, extra_edges, edge_ptr, max_sent_nnz) -> DepGraph:
    if edge_ptr is None:
        raise L.EdgError("extra_edges needs edge_ptr (int [B+1]: the pairs of sentence b are edge_ptr[b] .. [b+1] - 1)")
    if extra_edges.dim() != 2 or extra_edges.shape[1] != 2:
        raise L.EdgError(f"extra_edges must be [E, 2], got {tuple(extra_edges.shape)}")
    if edge_ptr.numel() != sent_ptr.numel():
        raise L.EdgError(f"edge_ptr has {edge_ptr.numel()} entries, sent_ptr {sent_ptr.numel()}")
    if max_len is None and not sent_ptr.is_cuda:
        sp = sent_ptr.to(torch.int64)
        max_len = int((sp[1:] - sp[:-1]).max()) if sp.numel() > 1 else 0
    heads = _i32(heads, device)
    sent_ptr = _i32(sent_ptr, device)
    edges = _i32(extra_edges, device)
    edge_ptr = _i32(edge_ptr, device)
    B, N, E = sent_ptr.numel() - 1, heads.numel(), edges.shape[0]
    if max_len is None:
        max_len = int((sent_ptr[1:] - sent_ptr[:-1]).max().item()) if B > 0 else 0
    row_ptr = torch.empty(N + 1, dtype=torch.int32, device=device)
    col = torch.empty(max(3 * N + 2 * E, 1), dtype=torch.int32, device=device)
    row_sent = torch.empty(max(N, 1), dtype=torch.int32, device=device)
    # in: the caller's bound (0 = none), out: the largest sentence
    smn = torch.full((1,), int(max_sent_nnz or 0), dtype=torch.int32, device=device)
    with torch.cuda.device(device):
        nbytes = L.load().edg_csr_from_heads_edges_workspace(B, N, E)
        ws = torch.empty(max(nbytes, 4), dtype=torch.uint8, device=device)
        L.call("edg_csr_from_heads_edges", L.ptr(heads), L.ptr(sent_ptr), L.ptr(edges) if E else None, L.ptr(edge_ptr),
               B, N, E, max_len, L.ptr(row_ptr), L.ptr(col), L.ptr(row_sent), L.ptr(smn), L.ptr(ws), ws.numel(),
               L.stream())
        if max_sent_nnz is None:
            max_sent_nnz = int(smn.item())          # one small device->host read
    return DepGraph(sent_ptr, row_ptr, col, row_sent[:N], B, N, max_len, max_sent_nnz=int(max_sent_nnz))


def graph_from_dense(adj: torch.Tensor, check: bool = True) -> DepGraph:
    """Dense ``[B,T,T]`` adjacency as the reference models receive it
    (``inputs['dependency_graph'][:, :T, :T]``, bert_amir5.py:589; any strides,
    float32 or int64) -> packed CSR over ``B*T`` rows.  Padding rows keep their
    self loop (graph.py:66) and therefore stay live single-node graphs.

    The kernels treat the adjacency as a 0/1 symmetric pattern (all graph.py can
    produce); ``check=True`` raises if the matrix holds other values."""
    if not adj.is_cuda:
        raise L.EdgError("graph_from_dense needs a CUDA tensor (there is no CPU path)")
    if adj.dim() != 3 or adj.shape[1] != adj.shape[2]:
        raise L.EdgError("adjacency must be [B,T,T]")
    if adj.dtype not in (torch.float32, torch.int64):
        adj = adj.float()
    B, T, _ = adj.shape
    rows = B * T
    dev = adj.device
    is64 = int(adj.dtype == torch.int64)
    row_ptr = torch.empty(rows + 1, dtype=torch.int32, device=dev)
    flags = torch.empty(2, dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        L.call("edg_csr_from_dense_count", L.ptr(adj), is64, B, T, adj.stride(0), adj.stride(1), adj.stride(2),
               L.ptr(row_ptr), L.ptr(flags), L.stream())
        # the largest CSR entry count of one sentence: any symmetric pattern is accepted, so the tree bound 3T - 2 that
        # DepGraph.tile_plan assumes otherwise does not hold (a dense sentence can overflow the fused kernels' tiles)
        sent_nnz = (row_ptr[T::T] - row_ptr[:rows:T]).max().view(1)
        host = torch.cat([row_ptr[rows:rows + 1], flags, sent_nnz]).cpu()     # one small device->host read
        nnz, odd, asym, max_sent_nnz = (int(v) for v in host)
        if check and (odd or asym):
            raise L.EdgError(
                f"dense adjacency is not a 0/1 symmetric pattern ({odd} non-binary, {asym} asymmetric entries); "
                "the CSR kernels implement graph.py:66-75 matrices only")
        col = torch.empty(max(nnz, 1), dtype=torch.int32, device=dev)
        L.call("edg_csr_from_dense_fill", L.ptr(adj), is64, B, T, adj.stride(0), adj.stride(1), adj.stride(2),
               L.ptr(row_ptr), L.ptr(col), L.stream())
    sent_ptr = torch.arange(0, rows + 1, T, dtype=torch.int32, device=dev)
    row_sent = torch.arange(B, dtype=torch.int32, device=dev).repeat_interleave(T)
    return DepGraph(sent_ptr, row_ptr, col, row_sent, B, rows, T, padded_T=T, max_sent_nnz=max_sent_nnz)


def tree_distance(graph: DepGraph, anchor_index: torch.Tensor, pad: Optional[str] = None,
                  T: Optional[int] = None, pairs: Optional[TriggerPairs] = None) -> torch.Tensor:
    """``get_dist_to_target`` (data_utils.py:319-323) for every sentence of the batch.

    ``pad=None`` -> packed int32 ``[N]``.  ``pad='max+1'`` (data_utils.py:486-488) or
    ``'zero'`` (:593-594) -> int64 ``[B,T]`` laid out like the collated
    ``dist_to_target`` column (data_utils.py:378).

    The kernel counts breadth-first hops.  On a graph with extra edges (``build_graph(..., extra_edges=...)``) it
    returns those hop counts; the reference's depth-first walk depends on the order it visits neighbours on a cycle and
    can over-estimate there (``tests/golden/tree_dist_cycle.npz``).  Where parity with the reference's distances
    matters, use the items' own ``dist_to_target`` (``PackedBatch.dist``).

    ``pairs`` (:class:`TriggerPairs`): ``anchor_index`` holds one anchor per pair, and the result is the per-pair packed
    ``int32 [pairs.n_pair_rows]`` (pair p's distances start at ``pairs.pair_row_ptr[p]``); ``pad`` must be None."""
    dev = graph.device
    anchor = _i32(anchor_index, dev)
    if pairs is not None:
        if pad is not None:
            raise L.EdgError("tree_distance(pairs=) returns the per-pair packed layout only (pad must be None)")
        if anchor.numel() != pairs.n_pairs:
            raise L.EdgError(f"expected {pairs.n_pairs} anchors (one per pair), got {anchor.numel()}")
        dist = torch.empty(max(pairs.n_pair_rows, 1), dtype=torch.int32, device=dev)
        with torch.cuda.device(dev):
            L.call("edg_tree_dist_pairs", L.ptr(graph.row_ptr), L.ptr(graph.col), L.ptr(graph.sent_ptr),
                   L.ptr(pairs.pair_sent), L.ptr(pairs.pair_row_ptr), L.ptr(anchor), pairs.n_pairs, graph.max_len,
                   L.ptr(dist), L.stream())
        return dist[:pairs.n_pair_rows]
    dist = torch.empty(max(graph.n_rows, 1), dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        L.call("edg_tree_dist", L.ptr(graph.row_ptr), L.ptr(graph.col), L.ptr(graph.sent_ptr), L.ptr(anchor),
               graph.n_graphs, graph.max_len, L.ptr(dist), L.stream())
        dist = dist[:graph.n_rows]
        if pad is None:
            return dist
        mode = {"max+1": L.PAD_MAX_PLUS_1, "zero": L.PAD_ZERO}[pad]
        T = T or graph.max_len
        out = torch.empty((graph.n_graphs, T), dtype=torch.int64, device=dev)
        L.call("edg_dist_pad", L.ptr(dist), L.ptr(graph.sent_ptr), graph.n_graphs, T, mode, L.ptr(out), L.stream())
    return out
