"""CPU checks of the packed route for dependency graphs that are not forests (CoreNLP enhanced dependencies): a
sentence travels as its breadth-first forest of heads plus the extra undirected edges a head array cannot hold
(wire.split_adjacency, collate_packed), synthetic batches gain such edges from a generator of their own
(synth.with_extra_edges), and sharding keeps them with their sentences."""
import numpy as np
import pytest
import torch

from oracle import ref_oracle as O
from test_host_cpu import _reference_items


def rebuild(heads, extra, n, size=None):
    """Dense 0/1 pattern of heads + extra edges (+ identity), as graph.py:66-75 builds it."""
    m = O.dense_adjacency_from_heads(heads, size or n)
    for i, j in np.asarray(extra).reshape(-1, 2):
        m[i, j] = m[j, i] = 1
    return m


def tree_plus_extras(n, n_extra, rng, size=100):
    from ed_gated_gcn_b200 import synth
    m = O.dense_adjacency_from_heads(synth.random_tree(n, rng), size)
    for _ in range(n_extra):
        i, j = rng.integers(0, n, 2)
        m[i, j] = m[j, i] = 1
    return m


def forest_plus_joins(rng, size=100):
    """Three trees side by side, then edges that join them (and one that closes a cycle across them)."""
    from ed_gated_gcn_b200 import synth
    parts = [synth.random_tree(k, rng) for k in (7, 5, 9)]
    heads, off = [], 0
    for p in parts:
        heads.append(np.where(p >= 0, p + off, -1))
        off += len(p)
    n = off
    m = O.dense_adjacency_from_heads(np.concatenate(heads), size)
    for i, j in ((0, 7), (8, 14), (3, 20)):
        m[i, j] = m[j, i] = 1
    return m, n


def hub(n, size=100):
    m = np.eye(size, dtype=np.int64)
    m[0, :n] = m[:n, 0] = 1
    m[n // 2, :n] = m[:n, n // 2] = 1          # a second hub closes cycles through the first
    return m


def check_split(m, n):
    import ed_gated_gcn_b200 as E
    heads, extra = E.split_adjacency(m, n)
    assert heads.dtype == np.int32 and heads.shape == (n,)
    assert extra.dtype == np.int32 and extra.ndim == 2 and extra.shape[1] == 2
    assert (extra[:, 0] < extra[:, 1]).all()
    keys = extra[:, 0].astype(np.int64) * n + extra[:, 1]
    assert (np.diff(keys) > 0).all()                                      # ascending, distinct
    got = rebuild(heads, extra, n, m.shape[0])
    want = m.copy()
    want[n:, :] = np.eye(m.shape[0], dtype=m.dtype)[n:, :]               # rows past n are padding: identity only
    want[:, n:] = np.eye(m.shape[0], dtype=m.dtype)[:, n:]
    assert np.array_equal(got[:n, :n] != 0, want[:n, :n] != 0)
    # no extra edge repeats a forest edge
    forest = {(min(i, int(h)), max(i, int(h))) for i, h in enumerate(heads) if h >= 0}
    assert not forest & {tuple(e) for e in extra.tolist()}
    return heads, extra


def test_split_adjacency_rebuilds_every_matrix():
    rng = np.random.default_rng(11)
    cases = [(tree_plus_extras(n, k, rng), n) for n in (2, 3, 10, 40, 100) for k in (0, 1, 5, 30)]
    cases += [forest_plus_joins(rng)]
    cases += [(np.eye(100, dtype=np.int64), 1), (np.eye(100, dtype=np.int64), 0)]
    cases += [(hub(n), n) for n in (2, 5, 60, 100)]
    dense = np.ones((100, 100), dtype=np.int64)                            # the complete graph on 100 tokens
    cases += [(dense, 100)]
    n_extra = 0
    for m, n in cases:
        _, extra = check_split(m, n)
        n_extra += len(extra)
    assert n_extra > 5000


def test_split_adjacency_on_forests_is_heads_from_adjacency():
    import ed_gated_gcn_b200 as E
    from ed_gated_gcn_b200 import synth
    rng = np.random.default_rng(12)
    for n in (1, 2, 7, 50, 100):
        for skewed in (False, True):
            m = O.dense_adjacency_from_heads(synth.random_tree(n, rng, skewed), 100)
            heads, extra = E.split_adjacency(m, n)
            assert np.array_equal(heads, E.heads_from_adjacency(m, n)) and extra.shape == (0, 2)
    m = np.eye(100, dtype=np.int64)
    for i, j in ((0, 3), (3, 5), (1, 2)):                                   # a forest of three components
        m[i, j] = m[j, i] = 1
    heads, extra = E.split_adjacency(m, 8)
    assert np.array_equal(heads, E.heads_from_adjacency(m, 8)) and extra.shape == (0, 2)
    # on a graph with cycles the forest is still the one heads_from_adjacency builds before it gives up
    m = tree_plus_extras(30, 10, rng)
    heads, extra = E.split_adjacency(m, 30)
    assert len(extra) > 0
    with pytest.raises(ValueError):
        E.heads_from_adjacency(m, 30)
    bfs = np.full(30, -2, dtype=np.int32)
    for root in range(30):                                                 # the breadth-first orientation, restated
        if bfs[root] != -2:
            continue
        bfs[root], frontier = -1, [root]
        while frontier:
            nxt = []
            for u in frontier:
                for v in np.nonzero(m[u, :30])[0]:
                    if v != u and bfs[v] == -2:
                        bfs[v] = u
                        nxt.append(int(v))
            frontier = nxt
    assert np.array_equal(heads, bfs)
    asym = np.eye(6, dtype=np.int64)
    asym[0, 1] = 1
    with pytest.raises(ValueError):
        E.split_adjacency(asym, 6)


def enhanced_items(seed=21, n_graphs=12, ori_ml=60):
    """Reference-format items whose adjacency carries enhanced-dependency-like extra edges on most sentences."""
    from ed_gated_gcn_b200 import synth
    batch = synth.with_extra_edges(synth.make_batch(n_graphs, 1, 40, seed=seed), rate=0.3, seed=seed + 1)
    rng = np.random.default_rng(seed + 2)
    pieces = [rng.integers(1, 4, size=int(n)).tolist() for n in batch.lengths]
    items = _reference_items(batch, pieces, ori_ml=ori_ml)
    for it, h, x in zip(items, batch.heads_list(), batch.extras_list()):
        it["dependency_graph"] = rebuild(h, x, len(h), ori_ml).tolist()
    return batch, items, pieces


def test_collate_packed_carries_enhanced_dependency_items():
    """At the parent commit collate_packed raised ValueError on the first item with an extra edge."""
    import ed_gated_gcn_b200 as E
    batch, items, pieces = enhanced_items()
    assert sum(len(x) > 0 for x in batch.extras_list()) >= 6
    pb = E.collate_packed(items)
    assert pb.n_graphs == 12 and pb.n_rows == batch.n_rows and pb.max_len == int(batch.lengths.max())
    assert pb.extra_edges.dtype == torch.int32 and pb.edge_ptr.dtype == torch.int32
    assert pb.edge_ptr.shape == (13,) and int(pb.edge_ptr[-1]) == pb.extra_edges.shape[0]
    want_nnz = 0
    for b, it in enumerate(items):
        lo, hi = batch.sent_ptr[b], batch.sent_ptr[b + 1]
        n = hi - lo
        h = pb.heads[lo:hi].numpy()
        x = pb.extra_edges[pb.edge_ptr[b]:pb.edge_ptr[b + 1]].numpy()
        m = np.asarray(it["dependency_graph"])
        assert np.array_equal(rebuild(h, x, n, 60)[:n, :n], m[:n, :n])
        assert pb.dist[lo:hi].tolist() == it["dist_to_target"][:n]
        start = pb.seg_start[lo:hi].numpy() - int(pb.piece_ptr[b])
        assert start.tolist() == (1 + np.concatenate([[0], np.cumsum(pieces[b])[:-1]])).tolist()
        assert pb.seg_len[lo:hi].tolist() == pieces[b]
        want_nnz = max(want_nnz, int((m[:n, :n] != 0).sum()))
    assert pb.max_sent_nnz == want_nnz
    dense_bytes = 12 * (60 * 60 * 4 + 60 * 90 * 4 + 60 * 8)
    assert pb.nbytes() < dense_bytes / 50
    moved = pb.to("cpu", non_blocking=False)                               # pin() / to() map every tensor field
    assert torch.equal(moved.extra_edges, pb.extra_edges)
    assert torch.equal(moved.edge_ptr, pb.edge_ptr) and moved.max_sent_nnz == pb.max_sent_nnz


def test_forest_batch_tensors_are_unchanged():
    import ed_gated_gcn_b200 as E
    from ed_gated_gcn_b200 import synth
    batch = synth.make_batch(12, 1, 40, seed=21)
    rng = np.random.default_rng(5)
    pieces = [rng.integers(1, 4, size=int(n)).tolist() for n in batch.lengths]
    items = _reference_items(batch, pieces)
    pb = E.collate_packed(items)
    assert pb.extra_edges is None and pb.edge_ptr is None
    heads = np.concatenate([E.heads_from_adjacency(it["dependency_graph"], it["sentence_length"]) for it in items])
    assert torch.equal(pb.heads, torch.from_numpy(heads))
    names = {k for k, v in vars(pb).items() if isinstance(v, torch.Tensor)}
    assert names == {"heads", "sent_ptr", "anchor", "dist", "polarity", "seg_start", "seg_len", "piece_ptr"}
    assert pb.nbytes() == sum(getattr(pb, k).numel() * getattr(pb, k).element_size() for k in names)
    assert pb.max_sent_nnz == max(3 * int(n) - 2 for n in batch.lengths)       # trees: n + 2 (n - 1)
    assert E.collate_packed([]).max_sent_nnz == 0


def test_with_extra_edges_leaves_the_tree_streams_alone():
    from ed_gated_gcn_b200 import synth
    a = synth.make_batch(64, 2, 30, seed=3)
    b = synth.with_extra_edges(synth.make_batch(64, 2, 30, seed=3), rate=0.5, seed=4)
    c = synth.make_batch(64, 2, 30, seed=3)
    for k in ("heads", "sent_ptr", "anchor", "lengths"):
        assert np.array_equal(getattr(a, k), getattr(b, k)) and np.array_equal(getattr(a, k), getattr(c, k))
        assert getattr(a, k).dtype == getattr(c, k).dtype
    assert a.extra_edges is None and a.edge_ptr is None
    assert b.edge_ptr.shape == (65,) and b.edge_ptr[-1] == len(b.extra_edges) > 50
    again = synth.with_extra_edges(a, rate=0.5, seed=4)
    assert np.array_equal(again.extra_edges, b.extra_edges) and np.array_equal(again.edge_ptr, b.edge_ptr)
    c2 = synth.config_batch("C2", n_graphs=64)
    assert np.array_equal(c2.heads, synth.config_batch("C2", n_graphs=64).heads)
    for h, x in zip(b.heads_list(), b.extras_list()):
        n = len(h)
        forest = {(min(i, int(p)), max(i, int(p))) for i, p in enumerate(h) if p >= 0}
        pairs = [tuple(e) for e in x.tolist()]
        assert all(0 <= i < j < n for i, j in pairs) and pairs == sorted(set(pairs)) and not forest & set(pairs)
        for i, j in pairs:                      # every extra edge closes a triangle with tree edges
            common = {int(h[i]), int(h[j])} | {k for k in range(n) if h[k] in (i, j)}
            assert any(((min(i, k), max(i, k)) in forest) and ((min(j, k), max(j, k)) in forest) for k in common)
    assert synth.with_extra_edges(a, rate=0.0).extra_edges.shape == (0, 2)


def test_shard_tree_batch_keeps_each_sentences_extra_edges():
    from ed_gated_gcn_b200 import parallel, synth
    batch = synth.with_extra_edges(synth.make_batch(21, 2, 25, seed=8), rate=0.4, seed=9)
    owned = []
    for rank in range(3):
        sub, idx = parallel.shard_tree_batch(batch, 3, rank)
        assert sub.edge_ptr.shape == (len(idx) + 1,) and sub.extra_edges.dtype == np.int32
        for k, b in enumerate(idx):
            assert np.array_equal(sub.extras_list()[k], batch.extras_list()[b])
            assert np.array_equal(sub.heads_list()[k], batch.heads_list()[b])
        owned += list(idx)
    assert sorted(owned) == list(range(21))
    plain, _ = parallel.shard_tree_batch(synth.make_batch(21, 2, 25, seed=8), 3, 0)
    assert plain.extra_edges is None and plain.edge_ptr is None
