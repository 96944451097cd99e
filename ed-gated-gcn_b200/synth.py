"""Synthetic dependency-tree batches (SURVEY.md 8d, "Synthetic inputs").

Host-side numpy only.  Used by the tests, ``bench.py`` and ``smoke()`` -- the
reference ships no data, so every input of the path is generated here from a
seed (default 14181, the reference's own ``--seed``, train.py:307).
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import List, Optional

import numpy as np

REFERENCE_SEED = 14181


def random_tree(n: int, rng: np.random.Generator, skewed: bool = False) -> np.ndarray:
    """Head indices (-1 = root) of a random tree over ``n`` tokens.

    Plain: random recursive tree (node i>0 attaches to U{0..i-1}) followed by a
    random relabelling, so heads are not ordered.  ``skewed``: one hub takes a
    child with probability 0.5, otherwise preferential attachment by degree+1
    (config 4: hub degree about n/2)."""
    heads = np.full(n, -1, dtype=np.int64)
    if n > 1:
        if not skewed:
            heads[1:] = (rng.random(n - 1) * np.arange(1, n)).astype(np.int64)
        else:
            deg = np.ones(n, dtype=np.float64)
            for i in range(1, n):
                if rng.random() < 0.5:
                    h = 0
                else:
                    w = deg[:i]
                    h = int(rng.choice(i, p=w / w.sum()))
                heads[i] = h
                deg[h] += 1.0
                deg[i] += 1.0
    perm = rng.permutation(n).astype(np.int32)   # old label -> new label
    out = np.full(n, -1, dtype=np.int32)
    kids = np.nonzero(heads >= 0)[0]
    out[perm[kids]] = perm[heads[kids]]
    return out


@dataclass
class TreeBatch:
    heads: np.ndarray        # int32 [N]   sentence-local head index, -1 = root
    sent_ptr: np.ndarray     # int32 [B+1] row offsets of the sentences
    anchor: np.ndarray       # int32 [B]   sentence-local trigger index
    lengths: np.ndarray      # int32 [B]
    extra_edges: Optional[np.ndarray] = None   # int32 [E,2] sentence-local (i, j), i < j: edges beyond the tree
    edge_ptr: Optional[np.ndarray] = None      # int32 [B+1] pairs of sentence b: edge_ptr[b] .. edge_ptr[b+1] - 1

    @property
    def n_graphs(self) -> int:
        return int(self.lengths.shape[0])

    @property
    def n_rows(self) -> int:
        return int(self.sent_ptr[-1])

    def heads_list(self) -> List[np.ndarray]:
        return [self.heads[self.sent_ptr[b]:self.sent_ptr[b + 1]] for b in range(self.n_graphs)]

    def extras_list(self) -> List[np.ndarray]:
        """Extra edges of every sentence (int32 [E_b, 2]; empty without extras)."""
        if self.extra_edges is None:
            return [np.zeros((0, 2), dtype=np.int32) for _ in range(self.n_graphs)]
        return [self.extra_edges[self.edge_ptr[b]:self.edge_ptr[b + 1]] for b in range(self.n_graphs)]


def make_batch(n_graphs: int, n_min: int, n_max: int, seed: int = REFERENCE_SEED,
               skewed: bool = False, lengths: Optional[np.ndarray] = None) -> TreeBatch:
    rng = np.random.default_rng(seed)
    if lengths is None:
        lengths = rng.integers(n_min, n_max + 1, size=n_graphs).astype(np.int32)
    else:
        lengths = np.asarray(lengths, dtype=np.int32)
    sent_ptr = np.zeros(n_graphs + 1, dtype=np.int32)
    np.cumsum(lengths, out=sent_ptr[1:])
    heads = np.empty(int(sent_ptr[-1]), dtype=np.int32)
    for b in range(n_graphs):
        heads[sent_ptr[b]:sent_ptr[b + 1]] = random_tree(int(lengths[b]), rng, skewed)
    anchor = (rng.random(n_graphs) * lengths).astype(np.int32)
    return TreeBatch(heads=heads, sent_ptr=sent_ptr, anchor=anchor, lengths=lengths)


DEFAULT_EXTRA_RATE = 0.1


def with_extra_edges(batch: TreeBatch, rate: float = DEFAULT_EXTRA_RATE, seed: int = REFERENCE_SEED) -> TreeBatch:
    """``batch`` plus edges like those CoreNLP's enhanced dependencies add to a tree (propagated conjunct subjects,
    controlled subjects): each token that has a head gets, with probability ``rate``, one extra edge to its
    grandparent or to a sibling, closing a triangle.  Edges are drawn from a generator of their own (``seed``), so the
    tree arrays -- which the result shares with ``batch`` -- and every seeded stream of ``make_batch`` stay as they
    are.  Per sentence the edges are distinct, never repeat a tree edge, and come as (i, j), i < j, in ascending order.

    The default rate is a synthetic choice: no statistic of real CoreNLP output was available to calibrate it."""
    rng = np.random.default_rng(seed)
    pairs = set()
    for b, h in enumerate(batch.heads_list()):
        cand = np.nonzero((h >= 0) & (rng.random(len(h)) < rate))[0]
        to_grandparent = rng.random(len(cand)) < 0.5
        for i, up in zip(cand.tolist(), to_grandparent.tolist()):
            p = int(h[i])
            sibs = np.nonzero(h == p)[0]
            sibs = sibs[sibs != i]
            if up and h[p] >= 0:
                j = int(h[p])
            elif len(sibs):
                j = int(sibs[rng.integers(len(sibs))])
            else:
                continue
            pairs.add((b, min(i, j), max(i, j)))
    rows = np.array(sorted(pairs), dtype=np.int32).reshape(-1, 3)
    edge_ptr = np.zeros(batch.n_graphs + 1, dtype=np.int32)
    np.cumsum(np.bincount(rows[:, 0], minlength=batch.n_graphs), out=edge_ptr[1:])
    return TreeBatch(heads=batch.heads, sent_ptr=batch.sent_ptr, anchor=batch.anchor, lengths=batch.lengths,
                     extra_edges=np.ascontiguousarray(rows[:, 1:]), edge_ptr=edge_ptr)


def candidate_pairs(batch: TreeBatch, per_sentence: Optional[int] = None, none_rate: float = 0.0,
                    seed: int = REFERENCE_SEED):
    """(sentence, candidate trigger) pairs over ``batch``, grouped by sentence, as ``(pair_ptr int32 [B+1], anchor int32
    [P])`` for ``graph.pairs_from_ptr``.  ``per_sentence=None``: every token of every sentence is a candidate, in token
    order (what the LitBank reader makes, data_utils.py:456-508).  Otherwise ``per_sentence`` anchors drawn uniformly
    with replacement (so anchors may repeat).  Each sentence gets no pairs with probability ``none_rate``; empty
    sentences never have any.  Draws come from a generator of their own (``seed``): every seeded stream of
    ``make_batch`` stays as it is."""
    rng = np.random.default_rng(seed)
    counts, anchors = [], []
    for n in batch.lengths.tolist():
        if n == 0 or (none_rate > 0 and rng.random() < none_rate):
            counts.append(0)
            continue
        a = np.arange(n, dtype=np.int32) if per_sentence is None else rng.integers(0, n, size=per_sentence).astype(np.int32)
        counts.append(len(a))
        anchors.append(a)
    pair_ptr = np.zeros(batch.n_graphs + 1, dtype=np.int32)
    np.cumsum(np.asarray(counts, dtype=np.int32), out=pair_ptr[1:])
    anchor = np.concatenate(anchors).astype(np.int32) if anchors else np.zeros(0, dtype=np.int32)
    return pair_ptr, anchor


# BASELINE.json configs (SURVEY.md 8d "Per-config shapes")
CONFIGS = {
    "C1": dict(n_graphs=32, n_min=5, n_max=50, D=300, L=2, C=34, dtype="f32", skewed=False),
    "C2": dict(n_graphs=4096, n_min=5, n_max=50, D=300, L=2, C=34, dtype="bf16", skewed=False),
    "C3": dict(n_graphs=16384, n_min=5, n_max=50, D=768, L=3, C=34, dtype="bf16", skewed=False),
    "C4": dict(n_graphs=1024, n_min=64, n_max=512, D=768, L=4, C=34, dtype="bf16", skewed=True),
    "C5": dict(n_graphs=65536, n_min=10, n_max=200, D=300, L=0, C=0, dtype="bf16", skewed=False),
}


def config_batch(name: str, n_graphs: Optional[int] = None, seed_offset: int = 0) -> TreeBatch:
    c = CONFIGS[name]
    idx = list(CONFIGS).index(name)
    return make_batch(n_graphs or c["n_graphs"], c["n_min"], c["n_max"],
                      seed=REFERENCE_SEED + idx + 1000 * seed_offset, skewed=c["skewed"])
