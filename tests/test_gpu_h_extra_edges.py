"""Dependency graphs that are not forests on the packed path: heads plus extra undirected edges -> CSR on the GPU
(edg_csr_from_heads_edges through graph.build_graph), bit for bit against an oracle CSR of the dense matrix, and the
gated-GCN stack on such graphs against the per-sentence oracle, on the fused layer kernel and on the unfused
kernels."""
import numpy as np
import pytest
import torch

from gpu_util import DEV, rel
from oracle import ref_oracle as O
from test_gpu_f_fused import check_tile_plan
from test_gpu_g_fused_limits import _run_stack, _spy_fused_plan
from test_host_extra_edges import enhanced_items, rebuild

pytestmark = pytest.mark.gpu


# ------------------------------------------------------------------------------------------------ helpers
def pack(heads_list, pairs_list):
    """Concatenated heads, sent_ptr, pairs [E,2] and edge_ptr (int32 numpy) of per-sentence heads and raw pairs."""
    lens = [len(h) for h in heads_list]
    sp = np.zeros(len(lens) + 1, dtype=np.int32)
    np.cumsum(lens, out=sp[1:])
    heads = np.concatenate([np.asarray(h, dtype=np.int32).reshape(-1) for h in heads_list] + [np.zeros(0, np.int32)])
    pairs = np.concatenate([np.asarray(p, dtype=np.int32).reshape(-1, 2) for p in pairs_list] + [np.zeros((0, 2), np.int32)])
    ep = np.zeros(len(lens) + 1, dtype=np.int32)
    np.cumsum([len(np.asarray(p).reshape(-1, 2)) for p in pairs_list], out=ep[1:])
    return heads, sp, pairs, ep


def dense_of(h, pairs):
    """graph.py:66-75 pattern of one sentence: tree (malformed heads = roots, as the kernels clean them) + the valid
    pairs (both endpoints inside the sentence)."""
    n = len(h)
    h = np.asarray(h, dtype=np.int64)
    clean = np.array([-1 if (x < 0 or x >= n or x == i or (h[x] == i and i > x)) else x for i, x in enumerate(h)], dtype=np.int64)
    p = np.asarray(pairs, dtype=np.int64).reshape(-1, 2)
    ok = (p >= 0).all(1) & (p < n).all(1)
    return rebuild(clean, p[ok], n) if n else np.zeros((0, 0), dtype=np.int64)


def oracle_csr(heads_list, pairs_list):
    row_ptr, col, row_sent, base, mx = [0], [], [], 0, 0
    for b, (h, p) in enumerate(zip(heads_list, pairs_list)):
        m = dense_of(h, p)
        for i in range(len(h)):
            col.extend(base + np.nonzero(m[i])[0])
            row_ptr.append(len(col))
            row_sent.append(b)
        mx = max(mx, int((m != 0).sum()))
        base += len(h)
    return (np.asarray(row_ptr, np.int32), np.asarray(col, np.int32), np.asarray(row_sent, np.int32), mx)


def build(heads_list, pairs_list, **kw):
    import ed_gated_gcn_b200 as E
    heads, sp, pairs, ep = pack(heads_list, pairs_list)
    return E.build_graph(torch.from_numpy(heads), torch.from_numpy(sp), device=DEV, extra_edges=torch.from_numpy(pairs),
                         edge_ptr=torch.from_numpy(ep), **kw)


def assert_csr(g, want):
    row_ptr, col, row_sent, mx = want
    assert np.array_equal(g.row_ptr.cpu().numpy(), row_ptr)
    assert np.array_equal(g.col[:len(col)].cpu().numpy(), col)
    assert np.array_equal(g.row_sent.cpu().numpy(), row_sent)
    assert g.max_sent_nnz == mx


def tree_dist_bfs(m, anchor):
    """Hop count + 1 from the anchor over the pattern m; 100001 where unreachable (the kernel's convention)."""
    n = len(m)
    d = np.full(n, -1)
    d[anchor] = 0
    front = [anchor]
    while front:
        nxt = []
        for u in front:
            for v in np.nonzero(m[u])[0]:
                if d[v] < 0:
                    d[v] = d[u] + 1
                    nxt.append(v)
        front = nxt
    return np.where(d >= 0, d + 1, O.UNREACHABLE + 1)


def random_pairs(n, k, rng):
    return rng.integers(0, n, size=(k, 2)) if n else np.zeros((0, 2), dtype=np.int64)


def messy_batch(rng):
    """Sentences that exercise the set semantics: every kind of redundant or invalid pair, in random order."""
    from ed_gated_gcn_b200 import synth
    H, P = [], []
    h = synth.random_tree(20, rng)
    kids = np.nonzero(h >= 0)[0]
    good = [(0, 5), (5, 0), (3, 17), (3, 17), (17, 3), (2, 9)]
    forest = [(int(k), int(h[k])) for k in kids[:4]] + [(int(h[k]), int(k)) for k in kids[4:8]]
    selfs = [(4, 4), (0, 0)]
    outside = [(-1, 3), (3, 20), (25, 2), (20, 20), (-5, -5), (7, 1 << 30)]
    p = np.array(good + forest + selfs + outside)
    H.append(h); P.append(p[rng.permutation(len(p))])
    H.append([]); P.append([])                                            # empty sentence
    H.append([-1]); P.append([(0, 0), (0, 1), (-1, 0)])                   # 1-token sentence, nothing valid
    H.append(synth.random_tree(30, rng)); P.append([])                    # no extras
    H.append([]); P.append([(0, 1)])                                      # empty sentence with a pair: dropped
    n = 50                                                                # hub row adjacent to every token
    h = synth.random_tree(n, rng)
    H.append(h); P.append([(7, j) for j in rng.permutation(n)] + [(j, 7) for j in range(0, n, 3)])
    H.append(synth.random_tree(40, rng)); P.append(random_pairs(40, 200, rng))     # dense: many duplicates
    h = np.array([3, 3, 5, -1, 9, 4, 0, 2, 2, 1], dtype=np.int32)            # malformed heads: self, mutual, out of range
    h[1], h[4], h[7] = 1, 12, -7
    H.append(h); P.append([(0, 3), (4, 5), (5, 4), (8, 9)])
    for n in (128, 512, 4096):                                            # long sentences
        H.append(synth.random_tree(n, rng)); P.append(random_pairs(n, n // 2, rng))
    H.append(synth.random_tree(300, rng)); P.append([(150, j) for j in range(300)])   # a hub in a long sentence
    return H, P


# ------------------------------------------------------------------------------------------------ CSR
def test_csr_is_the_dense_pattern_bit_for_bit():
    rng = np.random.default_rng(1)
    H, P = messy_batch(rng)
    want = oracle_csr(H, P)
    g = build(H, P)
    assert_csr(g, want)
    assert g.max_len == 4096 and g.max_sent_nnz > 600
    # the result is a set: the order of the pairs (and of their endpoints) does not matter
    P2 = [np.asarray(p).reshape(-1, 2)[rng.permutation(len(np.asarray(p).reshape(-1, 2)))][:, ::-1] for p in P]
    assert_csr(build(H, P2), want)
    # the bound the caller guarantees, exactly met
    assert_csr(build(H, P, max_len=4096, max_sent_nnz=want[3]), want)


def test_no_extra_edges_gives_the_bytes_of_csr_from_heads():
    import ed_gated_gcn_b200 as E
    from ed_gated_gcn_b200 import synth
    for batch in (synth.make_batch(300, 0, 50, seed=2), synth.make_batch(40, 100, 700, seed=3, skewed=True)):
        ref = E.build_graph(torch.from_numpy(batch.heads), torch.from_numpy(batch.sent_ptr), device=DEV)
        g = build(batch.heads_list(), [[] for _ in range(batch.n_graphs)])
        nnz = int(ref.row_ptr[-1])
        assert torch.equal(g.row_ptr, ref.row_ptr) and torch.equal(g.row_sent, ref.row_sent)
        assert torch.equal(g.col[:nnz], ref.col[:nnz]) and g.max_len == ref.max_len
        assert g.max_sent_nnz == max(3 * int(n) - 2 for n in batch.lengths if n)


def test_equal_length_batch_equals_graph_from_dense():
    import ed_gated_gcn_b200 as E
    from ed_gated_gcn_b200 import synth
    rng = np.random.default_rng(3)
    B, T = 64, 37
    H = [synth.random_tree(T, rng) for _ in range(B)]
    P = [random_pairs(T, int(rng.integers(0, 40)), rng) for _ in range(B)]
    adj = torch.from_numpy(np.stack([dense_of(h, p) for h, p in zip(H, P)]).astype(np.float32)).to(DEV)
    d = E.graph_from_dense(adj)
    g = build(H, P)
    nnz = int(d.row_ptr[-1])
    assert torch.equal(g.row_ptr, d.row_ptr) and torch.equal(g.col[:nnz], d.col[:nnz])
    assert torch.equal(g.row_sent, d.row_sent) and g.max_sent_nnz == d.max_sent_nnz


def test_device_max_sent_nnz_equals_the_packed_batch():
    import ed_gated_gcn_b200 as E
    _, items, _ = enhanced_items(seed=31, n_graphs=40)
    pb = E.collate_packed(items)
    g = E.build_graph(pb.heads, pb.sent_ptr, device=DEV, extra_edges=pb.extra_edges, edge_ptr=pb.edge_ptr)
    assert g.max_sent_nnz == pb.max_sent_nnz and g.max_len == pb.max_len
    n = [it["sentence_length"] for it in items]
    assert int(g.row_ptr[-1]) == sum(int((np.asarray(it["dependency_graph"])[:k, :k] != 0).sum()) for it, k in zip(items, n))


def test_build_with_both_bounds_is_captured_without_a_device_to_host_read():
    """With max_len and max_sent_nnz given, build_graph + tree_distance record into a CUDA graph (a device->host read
    during capture raises) and the replay gives the eager result."""
    import ed_gated_gcn_b200 as E
    from ed_gated_gcn_b200 import synth
    batch = synth.with_extra_edges(synth.config_batch("C2", n_graphs=512), rate=0.2, seed=5)
    H, P = batch.heads_list(), batch.extras_list()
    want = oracle_csr(H, P)
    st = {k: torch.from_numpy(v).to(DEV) for k, v in dict(h=batch.heads, sp=batch.sent_ptr, e=batch.extra_edges,
                                                           ep=batch.edge_ptr, a=batch.anchor).items()}
    max_len = int(batch.lengths.max())
    eager = E.build_graph(st["h"], st["sp"], max_len=max_len, extra_edges=st["e"], edge_ptr=st["ep"])
    d_eager = E.tree_distance(eager, st["a"])
    torch.cuda.synchronize()
    cg = torch.cuda.CUDAGraph()
    with torch.cuda.graph(cg):
        g = E.build_graph(st["h"], st["sp"], max_len=max_len, extra_edges=st["e"], edge_ptr=st["ep"],
                          max_sent_nnz=want[3])
        d = E.tree_distance(g, st["a"])
    cg.replay()
    torch.cuda.synchronize()
    assert_csr(g, want)
    assert torch.equal(d, d_eager)


def test_tree_distance_on_cyclic_graphs_is_bfs():
    import ed_gated_gcn_b200 as E
    rng = np.random.default_rng(6)
    H, P = messy_batch(rng)
    g = build(H, P)
    lens = np.array([len(h) for h in H])
    anchor = (rng.random(len(H)) * lens).astype(np.int32)
    got = E.tree_distance(g, torch.from_numpy(anchor).to(DEV)).cpu().numpy()
    want = np.concatenate([tree_dist_bfs(dense_of(h, p), int(a)) for h, p, a in zip(H, P, anchor) if len(h)])
    assert np.array_equal(got, want)


def test_tile_plan_invariants_with_extra_edges():
    import ed_gated_gcn_b200 as E
    from ed_gated_gcn_b200 import ops, synth
    batch = synth.with_extra_edges(synth.config_batch("C2", n_graphs=2000), rate=0.3, seed=7)
    g = E.build_graph(torch.from_numpy(batch.heads), torch.from_numpy(batch.sent_ptr), device=DEV,
                      extra_edges=torch.from_numpy(batch.extra_edges), edge_ptr=torch.from_numpy(batch.edge_ptr))
    for rows in (ops.fused_tile_rows(300, 300), 64):
        plan = g.tile_plan(rows)
        assert plan is not None
        check_tile_plan(batch.sent_ptr, g, rows, plan)


# ------------------------------------------------------------------------------------------------ stack level
def _stack_case(batch, dtype, seed):
    import ed_gated_gcn_b200 as E
    D, C, Lyr = 300, 34, 2
    torch.manual_seed(seed)
    stack = E.GatedGCNStack(D, n_layers=Lyr, n_classes=C, gate_arch="sig-2", compute_dtype=dtype).to(DEV)
    gen = torch.Generator().manual_seed(seed + 1)
    O.reference_init_(list(stack.parameters()), gen)
    dense = torch.nn.Linear(2 * D, C).to(DEV)
    graph = E.build_graph(torch.from_numpy(batch.heads), torch.from_numpy(batch.sent_ptr), device=DEV,
                          extra_edges=torch.from_numpy(batch.extra_edges), edge_ptr=torch.from_numpy(batch.edge_ptr))
    anchor = torch.from_numpy(batch.anchor).to(DEV)
    dist = E.tree_distance(graph, anchor)
    xp = torch.randn(batch.n_rows, D, generator=gen)
    targets = torch.arange(batch.n_graphs) % C
    dc = dist.cpu().long()
    sp = batch.sent_ptr
    sents = [(xp[sp[b]:sp[b + 1]], torch.from_numpy(dense_of(h, x)).float(), int(batch.anchor[b]), dc[sp[b]:sp[b + 1]])
             for b, (h, x) in enumerate(zip(batch.heads_list(), batch.extras_list()))]
    return stack, dense, graph, anchor, dist, xp, targets, sents, Lyr


def test_bf16_stack_with_extra_edges_vs_oracle_and_unfused(monkeypatch):
    from ed_gated_gcn_b200 import gated, synth
    from test_gpu_c_models import _check_routing, _compare, _oracle_run
    batch = synth.with_extra_edges(synth.config_batch("C2", n_graphs=160), rate=0.3, seed=8)
    assert len(batch.extra_edges) > 200
    stack, dense, graph, anchor, dist, xp, targets, sents, Lyr = _stack_case(batch, torch.bfloat16, 81)
    sp = batch.sent_ptr
    seen = _spy_fused_plan(monkeypatch)
    out, loss, dx = _run_stack(stack, dense, graph, xp.to(DEV), anchor, dist, targets)
    assert seen and seen[0] is not None                                    # the fused kernels ran
    ora = _oracle_run(stack, dense, sents, targets)
    tol = 2e-2
    assert rel(out.x_out, torch.cat(ora["x_out"])) < tol
    ora_g = _oracle_run(stack, dense, sents, targets, forced=_check_routing(out, ora, sp[:-1]))
    _compare(out, loss, dx, stack, dense, ora, ora_g, tol, Lyr)
    fused_logits, fused_x_out = out.logits.detach().clone(), out.x_out.detach().clone()
    monkeypatch.setattr(gated, "_FUSED", False)
    out_u, loss_u, dx_u = _run_stack(stack, dense, graph, xp.to(DEV), anchor, dist, targets)
    assert seen[-1] is None
    assert rel(out_u.logits, fused_logits) < tol and rel(out_u.x_out, fused_x_out) < tol
    ora_u = _oracle_run(stack, dense, sents, targets, forced=_check_routing(out_u, ora, sp[:-1]))
    _compare(out_u, loss_u, dx_u, stack, dense, ora, ora_u, tol, Lyr)


def test_fp32_stack_with_extra_edges_vs_oracle():
    from ed_gated_gcn_b200 import synth
    from test_gpu_c_models import _compare, _oracle_run
    batch = synth.with_extra_edges(synth.make_batch(24, 5, 50, seed=9), rate=0.4, seed=10)
    stack, dense, graph, anchor, dist, xp, targets, sents, Lyr = _stack_case(batch, torch.float32, 91)
    out, loss, dx = _run_stack(stack, dense, graph, xp.to(DEV), anchor, dist, targets)
    ora = _oracle_run(stack, dense, sents, targets)
    _compare(out, loss, dx, stack, dense, ora, ora, 1e-5, Lyr)


def test_sentence_over_512_entries_through_extra_edges_gets_no_tile_plan(monkeypatch):
    from ed_gated_gcn_b200 import ops, synth
    from test_gpu_c_models import _check_routing, _compare, _oracle_run
    rng = np.random.default_rng(12)
    base = synth.make_batch(10, 40, 48, seed=11)
    P = [np.zeros((0, 2), np.int32) for _ in range(base.n_graphs)]
    n3 = int(base.lengths[3])
    P[3] = np.argwhere(np.triu(rng.random((n3, n3)) < 0.5, 1)).astype(np.int32)       # about n^2 / 2 extra entries
    P[5] = random_pairs(int(base.lengths[5]), 10, rng).astype(np.int32)
    ep = np.zeros(base.n_graphs + 1, dtype=np.int32)
    np.cumsum([len(p) for p in P], out=ep[1:])
    batch = synth.TreeBatch(heads=base.heads, sent_ptr=base.sent_ptr, anchor=base.anchor, lengths=base.lengths,
                            extra_edges=np.concatenate(P), edge_ptr=ep)
    stack, dense, graph, anchor, dist, xp, targets, sents, Lyr = _stack_case(batch, torch.bfloat16, 121)
    nnz = [int((s[1] != 0).sum()) for s in sents]
    assert nnz[3] > 512 and max(np.delete(nnz, 3)) <= 512 and graph.max_sent_nnz == nnz[3]
    assert graph.tile_plan(ops.fused_tile_rows(300, 300)) is None
    seen = _spy_fused_plan(monkeypatch)
    out, loss, dx = _run_stack(stack, dense, graph, xp.to(DEV), anchor, dist, targets)
    assert seen == [None]
    ora = _oracle_run(stack, dense, sents, targets)
    ora_g = _oracle_run(stack, dense, sents, targets, forced=_check_routing(out, ora, batch.sent_ptr[:-1]))
    _compare(out, loss, dx, stack, dense, ora, ora_g, 2e-2, Lyr)


def test_packed_enhanced_items_drive_the_same_result_as_the_dense_batch():
    """Reference items with enhanced adjacency -> collate_packed -> pinned -> GPU -> heads + extra edges -> CSR gives
    the same layer output as the dense [B,T,T] adjacency of the same items through forward(text, adj)."""
    import ed_gated_gcn_b200 as E
    batch, items, _ = enhanced_items(seed=41, n_graphs=10)
    pb = E.collate_packed(items).pin().to(DEV)
    assert pb.extra_edges is not None and pb.extra_edges.is_cuda
    graph = E.build_graph(pb.heads, pb.sent_ptr, max_len=pb.max_len, extra_edges=pb.extra_edges, edge_ptr=pb.edge_ptr,
                          max_sent_nnz=pb.max_sent_nnz)
    T = pb.max_len
    adj = torch.tensor([it["dependency_graph"] for it in items], dtype=torch.float32)[:, :T, :T].to(DEV)
    layer = E.GraphConvolution(16, 16, None).to(DEV)
    torch.nn.init.xavier_uniform_(layer.weight); torch.nn.init.uniform_(layer.bias, -0.1, 0.1)
    x = torch.randn(10, T, 16, device=DEV)
    dense_out = layer(x, adj)
    rows = torch.cat([x[b, :int(n)] for b, n in enumerate(batch.lengths)])
    packed_out = E.gcn_layer(rows, graph, layer.weight, layer.bias)
    want = torch.cat([dense_out[b, :int(n)] for b, n in enumerate(batch.lengths)])
    assert rel(packed_out, want) < 1e-6
