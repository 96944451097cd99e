"""Packed wire format of a batch (SURVEY.md 8f N3).

The reference collates every sentence as Python lists into dense tensors -- ``dependency_graph``
``[B,100,100]`` fp32 (40 KB per sentence), ``transform`` ``[B,100,120]`` fp32 (48 KB), ``dist_to_target``
``[B,100]`` int64 (data_utils.py:362-402, ``tensor_type`` / ``collate_fn``) -- and copies them host->device
per batch (train.py:108).  The hot path only needs ~16 bytes per token:

    heads int32[N] (-1 = root), sent_ptr int32[B+1], anchor int32[B], dist int32[N] (optional: the GPU
    recomputes it), seg_start/seg_len int32[N] + piece_ptr int32[B+1] (word pieces of every word)

Dependency graphs that are not forests (CoreNLP enhanced dependencies add edges that close cycles) travel as their
breadth-first forest in ``heads`` plus the remaining edges, ``extra_edges`` int32[E,2] + ``edge_ptr`` int32[B+1]
(8 bytes per extra edge; both absent when every sentence is a forest).

The LitBank reader makes one item per (sentence, candidate trigger) pair, so a sentence arrives once per candidate.
``collate_packed(..., group_sentences=True)`` sends such a sentence once, with ``pair_ptr`` int32[S+1] grouping the
pairs by sentence; ``anchor``, ``polarity`` and ``dist`` are then per pair (``dist`` in the per-pair packed layout).

``collate_packed`` builds that from the reference's own per-sentence item dicts (host, numpy);
``PackedBatch.pin`` / ``.to`` move it with one small copy per field.  Host-side only: no kernels here.
"""
from __future__ import annotations

from dataclasses import dataclass, fields
from typing import Dict, List, Optional, Sequence

import numpy as np
import torch


def _bfs_heads(a: np.ndarray, n: int):
    """Heads of the breadth-first orientation of the boolean pattern ``a`` and the number of edges it holds."""
    heads = np.full(n, -2, dtype=np.int32)
    used = 0
    for root in range(n):
        if heads[root] != -2:
            continue
        heads[root] = -1
        frontier = [root]
        while frontier:
            nxt = []
            for u in frontier:
                for v in np.nonzero(a[u])[0]:
                    if v != u and heads[v] == -2:
                        heads[v] = u
                        used += 1
                        nxt.append(int(v))
            frontier = nxt
    return heads, used


def _pattern(adj, n: int) -> np.ndarray:
    a = np.asarray(adj)[:n, :n] != 0
    if not np.array_equal(a, a.T):
        raise ValueError("adjacency is not symmetric")
    return a


def heads_from_adjacency(adj, n: int) -> np.ndarray:
    """Orient the symmetric 0/1 matrix of graph.py:66-75 (first ``n`` rows/cols) as head indices: every
    connected component is rooted at its smallest token (-1), every other token points at the neighbour that
    discovered it in a breadth-first sweep.  The CSR built from these heads (self + parent + children) is the
    non-zero pattern of the matrix.  Raises ValueError when the matrix is not a forest (an edge would be lost;
    ``split_adjacency`` keeps such edges)."""
    a = _pattern(adj, n)
    heads, used = _bfs_heads(a, n)
    n_edges = (int(a.sum()) - int(np.trace(a))) // 2
    if used != n_edges:
        raise ValueError(f"adjacency is not a forest ({n_edges} edges, {used} fit a head array): "
                         "use split_adjacency or graph_from_dense")
    return heads


def split_adjacency(adj, n: int):
    """Any symmetric 0/1 matrix of graph.py:66-75 (first ``n`` rows/cols), e.g. one built from CoreNLP enhanced
    dependencies whose extra edges close cycles -> ``(heads, extra)``.  ``heads`` is the breadth-first forest
    ``heads_from_adjacency`` returns for every input; ``extra`` int32 ``[E_b, 2]`` holds the remaining edges as
    ``(i, j)`` with ``i < j``, in ascending order (empty for a forest).  The forest's CSR plus these edges
    (``graph.build_graph(..., extra_edges=...)``) is the non-zero pattern of the matrix.  Raises ValueError on an
    asymmetric matrix."""
    a = _pattern(adj, n)
    heads, _ = _bfs_heads(a, n)
    rest = np.triu(a, 1)
    kids = np.nonzero(heads >= 0)[0]
    par = heads[kids]
    rest[np.minimum(kids, par), np.maximum(kids, par)] = False
    return heads, np.argwhere(rest).astype(np.int32).reshape(-1, 2)


def segments_from_transform_rows(transform, n_words: int):
    """One sentence's ``[ORI_ML][BERT_ML]`` transform (data_utils.py:438-451) -> (start, len) per word."""
    t = np.asarray(transform, dtype=np.float32)[:n_words]
    nz = t != 0
    length = nz.sum(1).astype(np.int32)
    start = np.where(length > 0, nz.argmax(1), 0).astype(np.int32)
    return start, length


@dataclass
class PackedBatch:
    heads: torch.Tensor                 # int32 [N]
    sent_ptr: torch.Tensor              # int32 [B+1]
    anchor: torch.Tensor                # int32 [B]
    dist: Optional[torch.Tensor] = None        # int32 [N]   (data_utils.py:319-323 values, unpadded)
    polarity: Optional[torch.Tensor] = None    # int64 [B]
    seg_start: Optional[torch.Tensor] = None   # int32 [N]   rows of the packed word-piece matrix
    seg_len: Optional[torch.Tensor] = None     # int32 [N]
    piece_ptr: Optional[torch.Tensor] = None   # int32 [B+1] word-piece rows of sentence b ([CLS] .. [SEP])
    max_len: int = 0
    extra_edges: Optional[torch.Tensor] = None  # int32 [E,2] sentence-local (i, j), i < j: edges a head array cannot hold
    edge_ptr: Optional[torch.Tensor] = None     # int32 [B+1] pairs of sentence b; both None when no sentence has one
    max_sent_nnz: int = 0               # largest CSR entry count of one sentence: n_b + 2 (forest edges) + 2 E_b
    pair_ptr: Optional[torch.Tensor] = None    # int32 [S+1] pairs of sentence s (grouped batches; None otherwise)
    n_pair_rows: int = 0                # grouped batches: sum over the pairs of their sentence's length (= dist rows)

    @property
    def n_graphs(self) -> int:
        """Sentences of the batch (= items unless grouped)."""
        return self.anchor.numel() if self.pair_ptr is None else self.sent_ptr.numel() - 1

    @property
    def n_pairs(self) -> int:
        return self.anchor.numel()

    @property
    def n_rows(self) -> int:
        return self.heads.numel()

    def nbytes(self) -> int:
        return sum(t.numel() * t.element_size() for t in self._tensors().values())

    def _tensors(self) -> Dict[str, torch.Tensor]:
        return {f.name: getattr(self, f.name) for f in fields(self)
                if isinstance(getattr(self, f.name), torch.Tensor)}

    def _map(self, fn) -> "PackedBatch":
        kw = {f.name: getattr(self, f.name) for f in fields(self)}
        kw.update({k: fn(v) for k, v in self._tensors().items()})
        return PackedBatch(**kw)

    def pin(self) -> "PackedBatch":
        return self._map(lambda t: t.pin_memory())

    def to(self, device, non_blocking: bool = True) -> "PackedBatch":
        return self._map(lambda t: t.to(device, non_blocking=non_blocking))


def _sentence_key(it: dict):
    """What makes two items the same sentence: length, word-piece ids and the adjacency pattern.  None for an item
    without ``cls_text_sep_indices`` (never grouped)."""
    if "cls_text_sep_indices" not in it:
        return None
    n = int(it["sentence_length"])
    m = int(it.get("cls_text_sep_length", len(it["cls_text_sep_indices"])))
    ids = np.asarray(it["cls_text_sep_indices"])[:m]
    return n, m, ids, np.asarray(it["dependency_graph"])[:n, :n] != 0


def _same_sentence(a, b) -> bool:
    return (a is not None and b is not None and a[0] == b[0] and a[1] == b[1] and np.array_equal(a[2], b[2])
            and np.array_equal(a[3], b[3]))


def collate_packed(items: Sequence[dict], with_dist: bool = True, with_transform: bool = True,
                   group_sentences: bool = False) -> PackedBatch:
    """The packed counterpart of ``collate_fn`` (data_utils.py:381-402) over the same item dicts
    (keys ``dependency_graph``, ``anchor_index``, ``sentence_length``, ``dist_to_target``, ``transform``,
    ``cls_text_sep_length``, ``polarity``; data_utils.py:362-379).

    ``group_sentences=True``: CONSECUTIVE items holding the same sentence (equal ``sentence_length``,
    ``cls_text_sep_length``, ``cls_text_sep_indices[:length]`` and non-zero pattern of ``dependency_graph[:n, :n]``)
    become one sentence with several (sentence, trigger) pairs; items without ``cls_text_sep_indices`` are never
    merged.  Pairs keep the item order, so per-pair outputs line up with the items.  Sentence-level fields (heads,
    sent_ptr, extra edges, word-piece segments, max_len) then hold each sentence once; ``anchor`` and ``polarity`` are
    per pair, ``dist`` is per-pair packed, and ``pair_ptr`` groups the pairs (see ``graph.pairs_from_ptr``)."""
    heads: List[np.ndarray] = []
    extras: List[np.ndarray] = []
    lens, anchors, dists, pols = [], [], [], []
    seg_s, seg_n, piece_ptr = [], [], [0]
    max_sent_nnz = 0
    pair_counts: List[int] = []
    prev_key = None
    for it in items:
        n = int(it["sentence_length"])
        if group_sentences:
            key = _sentence_key(it)
            if pair_counts and _same_sentence(prev_key, key):
                pair_counts[-1] += 1
                anchors.append(int(it["anchor_index"]))
                if with_dist and "dist_to_target" in it:
                    dists.append(np.asarray(it["dist_to_target"][:n], dtype=np.int32))
                if "polarity" in it:
                    pols.append(int(it["polarity"]))
                continue
            prev_key = key
            pair_counts.append(1)
        h, x = split_adjacency(it["dependency_graph"], n)
        heads.append(h)
        extras.append(x)
        max_sent_nnz = max(max_sent_nnz, n + 2 * int((h >= 0).sum()) + 2 * len(x))
        lens.append(n)
        anchors.append(int(it["anchor_index"]))
        if with_dist and "dist_to_target" in it:
            dists.append(np.asarray(it["dist_to_target"][:n], dtype=np.int32))
        if "polarity" in it:
            pols.append(int(it["polarity"]))
        if with_transform and "transform" in it:
            s, l = segments_from_transform_rows(it["transform"], n)
            seg_s.append(s + piece_ptr[-1])
            seg_n.append(l)
            n_pieces = int(it["cls_text_sep_length"]) if "cls_text_sep_length" in it else int((s + l).max(initial=0)) + 1
            piece_ptr.append(piece_ptr[-1] + n_pieces)
    S = len(lens)
    sent_ptr = np.zeros(S + 1, dtype=np.int32)
    np.cumsum(np.asarray(lens, dtype=np.int32), out=sent_ptr[1:])
    t = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a, dtype=dt))
    cat = lambda xs, dt: t(np.concatenate(xs) if xs else np.zeros(0, dtype=dt), dt)
    n_extra = np.asarray([len(x) for x in extras], dtype=np.int32)
    edge_ptr = None
    if n_extra.sum() > 0:
        edge_ptr = np.zeros(S + 1, dtype=np.int32)
        np.cumsum(n_extra, out=edge_ptr[1:])
    pair_ptr = None
    n_pair_rows = 0
    if group_sentences:
        pair_ptr = np.zeros(S + 1, dtype=np.int32)
        np.cumsum(np.asarray(pair_counts, dtype=np.int32), out=pair_ptr[1:])
        n_pair_rows = int(np.dot(np.asarray(lens, dtype=np.int64), np.asarray(pair_counts, dtype=np.int64))) if S else 0
    return PackedBatch(
        heads=cat(heads, np.int32), sent_ptr=t(sent_ptr, np.int32), anchor=t(np.asarray(anchors), np.int32),
        dist=cat(dists, np.int32) if len(dists) == len(items) and items else None,
        polarity=t(np.asarray(pols), np.int64) if len(pols) == len(items) and items else None,
        seg_start=cat(seg_s, np.int32) if len(seg_s) == S and items else None,
        seg_len=cat(seg_n, np.int32) if len(seg_n) == S and items else None,
        piece_ptr=t(np.asarray(piece_ptr), np.int32) if len(seg_s) == S and items else None,
        max_len=int(max(lens)) if lens else 0,
        extra_edges=t(np.concatenate(extras), np.int32) if edge_ptr is not None else None,
        edge_ptr=t(edge_ptr, np.int32) if edge_ptr is not None else None,
        max_sent_nnz=max_sent_nnz,
        pair_ptr=t(pair_ptr, np.int32) if pair_ptr is not None else None, n_pair_rows=n_pair_rows)
