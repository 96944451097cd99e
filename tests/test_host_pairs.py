"""(sentence, candidate trigger) pairs on the host: grouping of consecutive items of one sentence in
``collate_packed(group_sentences=True)``, the per-pair ``dist`` layout, ``pairs_from_ptr`` on CPU tensors (layout and
input checks) and ``synth.candidate_pairs``."""
import numpy as np
import pytest
import torch

from oracle import ref_oracle as O
from test_host_cpu import _reference_items
from test_host_extra_edges import enhanced_items


def _items_per_candidate(batch, pieces, anchors_of, ori_ml=60):
    """One reference item per (sentence, anchor), in sentence order: what the LitBank reader produces."""
    items = []
    base = _reference_items(batch, pieces, ori_ml=ori_ml)
    for b, it in enumerate(base):
        ids = [101] + list(range(1000 + 7 * b, 1000 + 7 * b + sum(pieces[b]))) + [102]
        h = batch.heads_list()[b]
        for a in anchors_of(b):
            d = dict(it)
            d["anchor_index"] = int(a)
            d["dist_to_target"] = O.pad_distance(O.tree_distance_bfs(h, int(a)), ori_ml, "max+1")
            d["cls_text_sep_indices"] = ids + [0] * 5
            d["polarity"] = (b + int(a)) % 3
            items.append(d)
    return items


def _batch(seed=3, n=6):
    from ed_gated_gcn_b200 import synth
    batch = synth.make_batch(n, 1, 12, seed=seed)
    rng = np.random.default_rng(seed)
    pieces = [rng.integers(1, 3, size=int(k)).tolist() for k in batch.lengths]
    return batch, pieces


def test_adjacent_items_of_one_sentence_become_one_sentence_with_pairs():
    import ed_gated_gcn_b200 as E
    batch, pieces = _batch()
    items = _items_per_candidate(batch, pieces, lambda b: range(int(batch.lengths[b])))
    flat = E.collate_packed(items)
    assert flat.pair_ptr is None and flat.n_graphs == len(items)              # default call: one sentence per item
    pb = E.collate_packed(items, group_sentences=True)
    S = batch.n_graphs
    assert pb.n_graphs == S and pb.n_pairs == len(items)
    assert np.array_equal(pb.sent_ptr.numpy(), batch.sent_ptr)
    assert np.array_equal(pb.pair_ptr.numpy(), batch.sent_ptr)               # every token a candidate: pair_ptr = sent_ptr
    # pair order = item order; anchors, polarity and per-pair dist line up with the items
    assert pb.anchor.tolist() == [it["anchor_index"] for it in items]
    assert pb.polarity.tolist() == [it["polarity"] for it in items]
    assert pb.dist.numel() == pb.n_pair_rows == int((batch.lengths.astype(np.int64) ** 2).sum())
    assert np.array_equal(pb.dist.numpy(), flat.dist.numpy())                  # per-pair packed = the expanded layout
    # the sentence-level arrays equal those of one item per sentence
    one = E.collate_packed([items[int(batch.sent_ptr[b])] for b in range(S)])
    for k in ("heads", "sent_ptr", "seg_start", "seg_len", "piece_ptr"):
        assert torch.equal(getattr(pb, k), getattr(one, k)), k
    assert pb.max_len == one.max_len and pb.max_sent_nnz == one.max_sent_nnz


def test_non_adjacent_items_of_one_sentence_stay_apart():
    import ed_gated_gcn_b200 as E
    batch, pieces = _batch(seed=4, n=3)
    items = _items_per_candidate(batch, pieces, lambda b: [0, 0])
    reordered = [items[0], items[2], items[1], items[3], items[4], items[5]]   # s0, s1, s0, s1, s2, s2
    pb = E.collate_packed(reordered, group_sentences=True)
    assert pb.n_graphs == 5 and pb.pair_ptr.tolist() == [0, 1, 2, 3, 4, 6]


def test_items_differing_in_ids_length_or_graph_are_not_merged():
    import ed_gated_gcn_b200 as E
    batch, pieces = _batch(seed=5, n=1)
    while batch.lengths[0] < 3:
        batch, pieces = _batch(seed=int(batch.lengths[0]) + 50, n=1)
    a, b = _items_per_candidate(batch, pieces, lambda s: [0, 1])
    assert E.collate_packed([a, b], group_sentences=True).n_graphs == 1
    ids = dict(b)
    ids["cls_text_sep_indices"] = list(b["cls_text_sep_indices"])
    ids["cls_text_sep_indices"][1] += 1                                        # another word piece
    assert E.collate_packed([a, ids], group_sentences=True).n_graphs == 2
    pad = dict(b)
    pad["cls_text_sep_indices"] = list(b["cls_text_sep_indices"])
    pad["cls_text_sep_indices"][-1] = 9                                        # beyond cls_text_sep_length: ignored
    assert E.collate_packed([a, pad], group_sentences=True).n_graphs == 1
    g = dict(b)
    adj = np.asarray(b["dependency_graph"]).copy()
    n = int(b["sentence_length"])
    i, j = 0, n - 1
    adj[i, j] = adj[j, i] = 1 - adj[i, j]                                      # another graph on the same tokens
    g["dependency_graph"] = adj.tolist()
    assert E.collate_packed([a, g], group_sentences=True).n_graphs == 2
    val = dict(b)
    val["dependency_graph"] = (np.asarray(b["dependency_graph"]) * 2.0).tolist()   # same non-zero pattern
    assert E.collate_packed([a, val], group_sentences=True).n_graphs == 1
    bare = [{k: v for k, v in it.items() if k != "cls_text_sep_indices"} for it in (a, b)]
    assert E.collate_packed(bare, group_sentences=True).n_graphs == 2          # no ids: never merged


def test_grouping_keeps_extra_edges_per_sentence():
    import ed_gated_gcn_b200 as E
    batch, items, pieces = enhanced_items(seed=31, n_graphs=8)
    rep = []
    for b, it in enumerate(items):
        for a in sorted({0, int(batch.lengths[b]) - 1}):
            d = dict(it)
            d["anchor_index"] = a
            d["cls_text_sep_indices"] = [101, 7 + b, 102]
            d["cls_text_sep_length"] = 3
            rep.append(d)
    one = E.collate_packed(items)
    pb = E.collate_packed(rep, group_sentences=True)
    assert pb.n_graphs == batch.n_graphs
    assert pb.edge_ptr is not None and torch.equal(pb.edge_ptr, one.edge_ptr) and torch.equal(pb.extra_edges, one.extra_edges)
    assert pb.pair_ptr.tolist() == np.concatenate([[0], np.cumsum([len({0, int(n) - 1}) for n in batch.lengths])]).tolist()


def _cpu_graph(lengths):
    from ed_gated_gcn_b200.graph import DepGraph
    sp = torch.zeros(len(lengths) + 1, dtype=torch.int32)
    sp[1:] = torch.cumsum(torch.tensor(lengths, dtype=torch.int32), 0)
    N = int(sp[-1])
    return DepGraph(sp, torch.zeros(N + 1, dtype=torch.int32), torch.zeros(1, dtype=torch.int32), None, len(lengths), N,
                    max(lengths) if lengths else 0)


def test_pairs_from_ptr_layout():
    from ed_gated_gcn_b200.graph import pairs_from_ptr
    lengths = [3, 0, 5, 1, 4]
    g = _cpu_graph(lengths)
    pair_ptr = torch.tensor([0, 2, 2, 5, 5, 7])                 # sentence 1 (empty) and 3 have no pairs
    anchor = torch.tensor([2, 2, 0, 4, 4, 3, 0])                # repeated anchors
    tp = pairs_from_ptr(g, pair_ptr, anchor)
    assert tp.n_pairs == 7 and tp.n_sentences == 5
    assert tp.pair_sent.tolist() == [0, 0, 2, 2, 2, 4, 4]
    assert tp.pair_start.tolist() == [0, 0, 3, 3, 3, 9, 9]
    assert tp.pair_row_ptr.tolist() == [0, 3, 6, 11, 16, 21, 25, 29]
    assert tp.n_pair_rows == 29
    tp2 = pairs_from_ptr(g, pair_ptr, anchor, n_pair_rows=29)
    for k in ("pair_ptr", "pair_sent", "pair_start", "anchor", "pair_row_ptr"):
        assert torch.equal(getattr(tp, k), getattr(tp2, k)), k


@pytest.mark.parametrize("pair_ptr, anchor, what", [
    ([0, 2, 1, 3], [0, 0, 0], "monotonically"),
    ([0, 1, 2, 2], [0, 0, 0], "monotonically"),               # ends before P
    ([1, 1, 2, 3], [0, 0, 0], "monotonically"),
    ([0, 1, 2, 3], [0, 2, 0], "outside"),                      # sentence 1 has 2 tokens
    ([0, 1, 2, 3], [-1, 0, 0], "outside"),
    ([0, 1, 3], [0, 0, 0], r"\[S\+1\]"),
])
def test_pairs_from_ptr_rejects_bad_input(pair_ptr, anchor, what):
    import ed_gated_gcn_b200 as E
    from ed_gated_gcn_b200.graph import pairs_from_ptr
    g = _cpu_graph([3, 2, 4])
    with pytest.raises(E.EdgError, match=what):
        pairs_from_ptr(g, torch.tensor(pair_ptr), torch.tensor(anchor))


def test_candidate_pairs():
    from ed_gated_gcn_b200 import synth
    batch = synth.make_batch(40, 0, 9, seed=12)
    assert (batch.lengths == 0).any()
    before = synth.make_batch(40, 0, 9, seed=12)
    pp, an = synth.candidate_pairs(batch)
    assert np.array_equal(pp, batch.sent_ptr)                   # all tokens
    assert np.array_equal(an, np.concatenate([np.arange(n) for n in batch.lengths]))
    pp, an = synth.candidate_pairs(batch, per_sentence=6, seed=3)
    cnt = np.diff(pp)
    assert ((cnt == 6) | (batch.lengths == 0)).all() and (cnt[batch.lengths == 0] == 0).all()
    owner = np.repeat(np.arange(batch.n_graphs), cnt)
    assert (an < batch.lengths[owner]).all() and (an >= 0).all()
    assert any(len(set(an[pp[s]:pp[s + 1]].tolist())) < cnt[s] for s in range(batch.n_graphs))   # repeated anchors
    pp2, an2 = synth.candidate_pairs(batch, per_sentence=6, seed=3)
    assert np.array_equal(pp, pp2) and np.array_equal(an, an2)
    pp, _ = synth.candidate_pairs(batch, none_rate=0.5, seed=4)
    assert ((np.diff(pp) == 0) & (batch.lengths > 0)).any()
    again = synth.make_batch(40, 0, 9, seed=12)                 # the batch stream is untouched
    assert np.array_equal(before.heads, again.heads) and np.array_equal(before.anchor, again.anchor)
