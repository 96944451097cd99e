"""The fused layer kernel (edg_gcn_fused.cu) at the limits of its tiles, and edg_head_du, against fp64 references over
EVERY sentence of the batch.

The limits under test:
  - a tile holds at most rows_cap (128) rows, 6 sentences and 512 CSR entries;
  - the kernel stages slot 0 = the row itself + 7 other neighbours per row, reads the second half of that word only
    above 4 entries and the global CSR above 8.
The batches are built from explicit head arrays: hubs with exactly k CSR entries (k = 4, 5, 8, 9, 16, 17, 64,
rows_cap) whose own entry sits in the first, a middle and the last slot of their CSR row; sentences that fill a tile
exactly (rows, sentences, both); runs of 1-token sentences; empty sentences inside tiles; a path of rows_cap tokens;
and one hub sentence per tile for the first 148 tiles followed by > 300 ordinary tiles, so every CTA of the persistent
grid moves from a hub tile to ordinary ones."""
import numpy as np
import pytest
import scipy.sparse as sps
import torch

from gpu_util import DEV, rel
from oracle import ref_oracle as O
from test_gpu_f_fused import check_tile_plan

pytestmark = pytest.mark.gpu

N_SM = 148
ROWS_CAP = 128
HUB_K = (4, 5, 8, 9, 16, 17, 64)          # + rows_cap


# ------------------------------------------------------------------------------------------------ graph builders
def hub_tree(n, k, pos, rng):
    """Heads of an n-token tree whose token ``pos`` has exactly k CSR entries (itself + k - 1 children).  As many
    children as possible lie below ``pos`` for pos = n - 1 (own entry last in the CSR row), none for pos = 0 (first),
    about half otherwise; the children are drawn at random, so their ids are not contiguous.  The other tokens form a
    chain hanging off one child."""
    assert 2 <= k <= n and 0 <= pos < n
    others = np.delete(np.arange(n), pos)
    below, above = others[others < pos], others[others > pos]
    nb = min(max((k - 1) // 2, k - 1 - len(above)), len(below))
    kids = np.concatenate([rng.choice(below, nb, replace=False), rng.choice(above, k - 1 - nb, replace=False)])
    heads = np.full(n, -1, dtype=np.int32)
    heads[kids] = pos
    prev = int(kids[rng.integers(len(kids))])
    for r in rng.permutation(np.setdiff1d(others, kids)):
        heads[r] = prev
        prev = int(r)
    return heads


def entries(heads):
    """CSR entries per row of one sentence: self + parent + children."""
    h = np.asarray(heads, dtype=np.int64)
    return 1 + (h >= 0) + np.bincount(h[h >= 0], minlength=len(h))


def ordinary_tree(n, rng, max_entries=16):
    """A random recursive tree (relabelled) with no row above ``max_entries`` entries."""
    from ed_gated_gcn_b200 import synth
    while True:
        h = synth.random_tree(n, rng)
        if n == 0 or entries(h).max() <= max_entries:
            return h


def path(n):
    return np.arange(-1, n - 1, dtype=np.int32)


def make_tree_batch(heads_list, rng):
    from ed_gated_gcn_b200 import synth
    lengths = np.array([len(h) for h in heads_list], dtype=np.int32)
    sp = np.zeros(len(lengths) + 1, dtype=np.int32)
    np.cumsum(lengths, out=sp[1:])
    heads = np.concatenate([np.asarray(h, dtype=np.int32) for h in heads_list]) if sp[-1] else np.zeros(0, np.int32)
    anchor = (rng.random(len(lengths)) * lengths).astype(np.int32)
    return synth.TreeBatch(heads=heads, sent_ptr=sp, anchor=anchor, lengths=lengths)


def limits_batch(R, seed=0):
    rng = np.random.default_rng(seed)
    sents = []
    # (a) the first 148 tiles: one hub (> 16 entries) sentence of >= 65 rows each -- two of them never share a tile,
    # so with 148 / n_split CTAs per column half every CTA's first tiles hold a hub
    for t in range(N_SM):
        k = (17, 24, 64, R, 33)[t % 5]
        n = int(rng.integers(max(k, 65), R + 1))
        sents.append(hub_tree(n, k, (0, n // 2, n - 1)[t % 3], rng))
    # (b) rows of exactly k entries, own entry in the first, a middle and the last slot
    for k in HUB_K + (R,):
        for which in range(3):
            n = int(rng.integers(k, R + 1))
            sents.append(hub_tree(n, k, (0, n // 2, n - 1)[which], rng))
    # (c) tile capacity: a full sentence; lengths adding up to rows_cap (3 and 6 sentences); a run of 1-token sentences
    # past the 6-sentence cap; a full sentence then a 1-token one; empty sentences inside a tile; a path of rows_cap
    for lens in ([R], [50, 40, R - 90], [30, 20, 25, 15, 10, R - 100], [1] * 13, [R, 1], [10, 0, 20, 0, 0, 5, 0]):
        sents += [ordinary_tree(n, rng) for n in lens]
    sents += [path(R), ordinary_tree(R, rng), [], []]
    # (d) ordinary tiles after the hub tiles: trees of <= 16 entries per row, some with rows of 5..16 entries
    for i in range(600):
        n = int(rng.integers(1, R + 1)) if i % 4 else int(rng.integers(40, R + 1))
        if i % 7 == 0 and n >= 16:
            sents.append(hub_tree(n, int(rng.choice([5, 8, 9, 12, 16])), int(rng.integers(n)), rng))
        else:
            sents.append(ordinary_tree(n, rng))
    return make_tree_batch(sents, rng)


_BATCHES = {}


def limits_setup(K, Nout):
    """(batch, graph, rows, plan) for the kernel's tile height, checked to be rows_cap."""
    import ed_gated_gcn_b200 as E
    from ed_gated_gcn_b200 import ops
    R = ROWS_CAP
    rows = ops.fused_tile_rows(K, Nout)
    assert rows == R, (K, Nout, rows)
    if R not in _BATCHES:
        _BATCHES[R] = limits_batch(R)
    batch = _BATCHES[R]
    g = E.build_graph(torch.from_numpy(batch.heads), torch.from_numpy(batch.sent_ptr), device=DEV)
    plan = g.tile_plan(rows)
    assert plan is not None
    return batch, g, rows, plan


def row_sent(batch):
    return np.repeat(np.arange(batch.n_graphs), batch.lengths)


def adj_hat(batch):
    """A^ = A / (rowsum + 1) over the whole batch as a sparse fp64 matrix, A from the oracle (gcn.py:35, 41)."""
    r, c = [], []
    for b, h in enumerate(batch.heads_list()):
        if len(h):
            i, j = np.nonzero(O.dense_adjacency_from_heads(h, len(h)))
            r.append(i + batch.sent_ptr[b]); c.append(j + batch.sent_ptr[b])
    N = batch.n_rows
    A = sps.csr_matrix((np.ones(sum(len(x) for x in r)), (np.concatenate(r), np.concatenate(c))), shape=(N, N))
    return sps.diags(1.0 / (np.asarray(A.sum(1)).ravel() + 1)) @ A


def hub_rows(batch, min_entries=9):
    """Global row of each sentence's row with the most CSR entries (-1 where none has >= min_entries)."""
    out = np.full(batch.n_graphs, -1, dtype=np.int64)
    for b, h in enumerate(batch.heads_list()):
        if len(h):
            e = entries(h)
            if e.max() >= min_entries:
                out[b] = batch.sent_ptr[b] + int(e.argmax())
    return out


def assert_rows_close(got, want, mag, what):
    """Element-wise bar of a bf16 aggregation: the staged rows and the output are each rounded once to bf16 (unit
    roundoff 2^-8; once more for a patched entry), so |got - want| <= 2^-8 (|A^| |terms| + |want|) up to fp32 terms;
    8e-3 = 2 x 2^-8.  Unlike a bar relative to the whole tensor, this catches one missing or wrong neighbour of a
    128-entry hub row."""
    got = got.double().cpu().numpy()
    err = np.abs(got - want)
    bound = 8e-3 * (mag + np.abs(want)) + 1e-5 * np.abs(want).max()
    bad = np.argwhere(err > bound)
    assert len(bad) == 0, f"{what}: {len(bad)} entries off, first (row, col) {tuple(bad[0])}: {err[tuple(bad[0])]:.3g} > {bound[tuple(bad[0])]:.3g}"


def inputs(batch, K, Nout, seed):
    from ed_gated_gcn_b200 import ops
    gen = torch.Generator().manual_seed(seed)
    x = torch.randn(batch.n_rows, K, generator=gen)
    w = torch.randn(Nout, K, generator=gen) / K ** 0.5
    bias = torch.randn(Nout, generator=gen)
    xr, wr = ops.as_rows(x.to(DEV), torch.bfloat16), ops.as_rows(w.to(DEV), torch.bfloat16)
    u = (xr.float().cpu().double() @ wr.float().cpu().double().t()).numpy()
    return xr, wr, bias, u


# ------------------------------------------------------------------------------------------------ tile plan
def test_tile_plan_at_the_limits():
    batch, g, rows, plan = limits_setup(300, 300)
    sp = batch.sent_ptr
    info = check_tile_plan(sp, g, rows, plan)
    nt = len(info)
    assert nt >= 3 * N_SM, nt
    # the batch reaches what it was built for
    ent = np.concatenate([entries(h) for h in batch.heads_list() if len(h)])
    ent_tile = [ent[info[t, 2]:info[t, 3]] for t in range(nt)]
    assert all(e.max() > 16 for e in ent_tile[:N_SM])                      # every CTA starts on hub tiles ...
    assert sum(e.max() <= 16 for e in ent_tile[N_SM:]) >= 2 * N_SM          # ... and goes on to ordinary ones
    nrow, nsent = info[:, 3] - info[:, 2], info[:, 1] - info[:, 0]
    assert (nrow == rows).sum() >= 5 and ((nrow == rows) & (nsent == 6)).any() and ((nrow == rows) & (nsent == 3)).any()
    assert ((nsent == 6) & (nrow == 6)).any()                                # six 1-token sentences
    lens = batch.lengths
    assert any((lens[info[t, 0]:info[t, 1]] == 0).any() and nrow[t] > 0 for t in range(nt))
    assert set(int(e) for e in ent) >= {4, 5, 8, 9, 16, 17, 64, rows}


# ------------------------------------------------------------------------------------------------ edg_gcn_layer
@pytest.mark.parametrize("shape", [(300, 300), (320, 320), (64, 64), (300, 161), (20, 300)])
def test_layer_forward_and_pool_at_the_limits(shape):
    from ed_gated_gcn_b200 import ops
    K, Nout = shape
    batch, g, rows, plan = limits_setup(K, Nout)
    xr, wr, bias, u = inputs(batch, K, Nout, seed=K + Nout)
    y, hmax, harg, _ = ops.gcn_layer(xr, wr, bias.to(DEV), g, 0, plan, rows, want_pool=True)
    ah = adj_hat(batch)
    want = ah @ u + bias.double().numpy()
    assert rel(y.float(), want) < 8e-3
    assert_rows_close(y.float(), want, abs(ah) @ np.abs(u), "y")
    base = y.as_strided((y.shape[0], y.stride(0)), (y.stride(0), 1))
    assert torch.isfinite(base.float()).all() and (base[:, Nout:] == 0).all()
    # the pool: exact column maximum of the STORED bf16 rows, first row on ties; empty sentences give 0 / -1
    yc = y.float().cpu().numpy()
    sp, lens = batch.sent_ptr, batch.lengths
    hm, ha = hmax.cpu().numpy(), harg.cpu().numpy()
    live = lens > 0
    m = np.maximum.reduceat(yc, sp[:-1][live], axis=0)
    assert np.array_equal(hm[live], m)
    rs = row_sent(batch)
    ridx = np.where(yc == hm[rs], np.arange(batch.n_rows)[:, None], np.iinfo(np.int64).max)
    assert np.array_equal(ha[live].astype(np.int64), np.minimum.reduceat(ridx, sp[:-1][live], axis=0))
    assert (hm[~live] == 0).all() and (ha[~live] == -1).all()


@pytest.mark.parametrize("shape", [(300, 300), (64, 64), (300, 161)])
def test_layer_adjoint_patch_and_colsum_at_the_limits(shape):
    from ed_gated_gcn_b200 import ops
    K, Nout = shape
    batch, g, rows, plan = limits_setup(K, Nout)
    xr, wr, _, u = inputs(batch, K, Nout, seed=3 * K + Nout)
    B = batch.n_graphs
    rng = np.random.default_rng(K + Nout)
    lens, starts = batch.lengths.astype(np.int64), batch.sent_ptr[:-1].astype(np.int64)
    pv = rng.standard_normal((B, Nout)).astype(np.float32)
    pa = (rng.random((B, Nout)) * lens[:, None]).astype(np.int64) + starts[:, None]
    hub = hub_rows(batch)
    on_hub = (hub[:, None] >= 0) & (rng.random((B, Nout)) < 0.5)           # half the columns of a hub sentence: the hub
    pa = np.where(on_hub, hub[:, None], pa)
    pa[rng.random((B, Nout)) < 0.2] = -1
    pa[lens == 0] = -1
    assert on_hub.sum() > 1000
    patched = u.copy()
    bi, ci = np.nonzero(pa >= 0)
    np.add.at(patched, (pa[bi, ci], ci), pv[bi, ci].astype(np.float64))
    aht = adj_hat(batch).T.tocsr()
    want, want_plain = aht @ patched, aht @ u
    y, _, _, cs = ops.gcn_layer(xr, wr, None, g, 1, plan, rows,
                                patch=(torch.from_numpy(pv).to(DEV), torch.from_numpy(pa).int().to(DEV)), want_colsum=True)
    assert rel(y.float(), want) < 8e-3
    assert_rows_close(y.float(), want, abs(aht) @ (np.abs(u) + np.abs(patched)), "y (patched)")
    assert rel(cs, patched.sum(0)) < 5e-3
    y0, _, _, cs0 = ops.gcn_layer(xr, wr, None, g, 1, plan, rows, want_colsum=True)
    assert rel(y0.float(), want_plain) < 8e-3
    assert_rows_close(y0.float(), want_plain, abs(aht) @ np.abs(u), "y")
    assert rel(cs0, u.sum(0)) < 5e-3
    base = y0.as_strided((y0.shape[0], y0.stride(0)), (y0.stride(0), 1))
    assert torch.isfinite(base.float()).all() and (base[:, Nout:] == 0).all()


# ------------------------------------------------------------------------------------------------ edg_head_du
@pytest.mark.parametrize("D", [300, 64])
def test_head_du_at_the_limits(D):
    """edg_head_du on the same tiles, with the arg-max rows of hub sentences on the hub (phase 4 then scatters into a
    row list longer than 8): against head_bwd -> aggregate (mode 1) and against the fp64 definition on every sentence."""
    import ed_gated_gcn_b200 as E
    from ed_gated_gcn_b200 import ops
    batch, g, rows, plan = limits_setup(D, D)
    B, N = batch.n_graphs, batch.n_rows
    gen = torch.Generator().manual_seed(D)
    h = ops.as_rows(torch.randn(N, D, generator=gen).to(DEV), torch.bfloat16)
    gate = torch.rand(B, D, generator=gen).to(DEV) * 0.9 + 0.05
    v = (torch.randn(B, D, generator=gen) * 0.2).to(DEV)
    c = torch.randn(B, generator=gen).to(DEV)
    gp = torch.randn(B, D, generator=gen).to(DEV)
    anchor = torch.from_numpy(batch.anchor).to(DEV)
    dist = E.tree_distance(g, anchor)
    scores, kl_b, kl, dvu, dcu, uu, sfu = ops.scores_kl_fwd(h, g, gate, v, c, dist, want_units=True, want_rows=True)
    _, arg_all = ops.pool_fwd(h, g, torch.ones((1, B, D), dtype=torch.float32, device=DEV))
    arg = arg_all[0].cpu().long()
    hub = torch.from_numpy(hub_rows(batch))
    on_hub = (hub[:, None] >= 0) & (torch.rand(B, D, generator=gen) < 0.5)
    arg = torch.where(on_hub, hub[:, None].expand(B, D), arg)
    hc = h.float().cpu()
    live = arg >= 0
    hmax = torch.where(live, hc[arg.clamp_min(0), torch.arange(D)[None, :]], torch.zeros(()))
    arg, hmax = arg.int().to(DEV), hmax.to(DEV)
    g_kl = torch.tensor(0.37, device=DEV)
    dh, dgate_ref, _, _ = ops.head_bwd(h, g, gate, v, dist, scores, kl_b, g_kl, None, gp, arg, None, want_dh=True, want_dv=False)
    du, db, dgate = ops.head_du(uu, g_kl, None, gate, v, gp, arg, sfu, hmax, g, plan)
    assert rel(du.float(), ops.aggregate(dh, g, mode=1, out_dtype=torch.float32)) < 8e-3
    assert rel(db, dh.float().sum(0)) < 5e-3
    assert rel(dgate, dgate_ref) < 1e-4
    base = du.as_strided((N, du.stride(0)), (du.stride(0), 1))
    assert torch.isfinite(base.float()).all() and (base[:, D:] == 0).all()
    # fp64 definition: dh_L[t] = g_kl u_t (g o v)_b + [t == arg(b,:)] (g o gp)_b,  du_L = A^T dh_L
    rs = row_sent(batch)
    q = (gate * v).double().cpu().numpy()
    dh64 = (0.37 * uu.double().cpu().numpy())[:, None] * q[rs]
    a = arg.cpu().long().numpy()
    bi, ci = np.nonzero(a >= 0)
    np.add.at(dh64, (a[bi, ci], ci), (gate * gp).double().cpu().numpy()[bi, ci])
    aht = adj_hat(batch).T.tocsr()
    want = aht @ dh64
    assert rel(du.float(), want) < 8e-3
    assert_rows_close(du.float(), want, abs(aht) @ np.abs(dh64), "du")


# ------------------------------------------------------------------------------------------------ stack level
def _stack_batch(R, seed=5):
    """~60 sentences at the limits: 90..rows_cap tokens, hubs of 9 to rows_cap entries, 1-token sentences."""
    rng = np.random.default_rng(seed)
    sents = []
    for i in range(48):
        n = R if i < 2 else int(rng.integers(90, R + 1))
        if i % 2 == 0:
            k = (9, 17, 40, n)[(i // 2) % 4]
            sents.append(hub_tree(n, k, (0, n // 2, n - 1)[i % 3], rng))
        else:
            sents.append(ordinary_tree(n, rng))
        if i % 4 == 3:
            sents.append(np.array([-1], dtype=np.int32))
    return make_tree_batch(sents, rng)


def _run_stack(stack, dense, graph, x0, anchor, dist, targets):
    for p in list(stack.parameters()) + list(dense.parameters()):
        p.grad = None
    x = x0.clone().requires_grad_(True)
    out = stack(x, graph, anchor, dist, lambda a, p: dense(torch.cat([a, p], 1)), head_params=list(dense.parameters()),
                return_x_out=True)
    loss = torch.nn.functional.cross_entropy(out.logits, targets.to(DEV)) + 0.01 * out.xy + 0.01 * out.kl
    loss.backward()
    return out, loss, x.grad


def _spy_fused_plan(monkeypatch):
    from ed_gated_gcn_b200 import gated
    seen, orig = [], gated._fused_plan

    def spy(*a):
        seen.append(orig(*a))
        return seen[-1]
    monkeypatch.setattr(gated, "_fused_plan", spy)
    return seen


def test_stack_at_the_tile_limits_vs_oracle_and_unfused(monkeypatch):
    """bf16 GatedGCNStack (D = 300, L = 2) on sentences of 90..rows_cap tokens with hubs and 1-token sentences: the fused
    path against the oracle (gradients under its own max-pool routing), then the unfused kernels on the same inputs."""
    import ed_gated_gcn_b200 as E
    from ed_gated_gcn_b200 import gated
    from test_gpu_c_models import _check_routing, _compare, _oracle_run
    R = ROWS_CAP
    batch = _stack_batch(R)
    assert batch.lengths.max() == R
    D, C, B, Lyr = 300, 34, batch.n_graphs, 2
    torch.manual_seed(77)
    stack = E.GatedGCNStack(D, n_layers=Lyr, n_classes=C, gate_arch="sig-2", compute_dtype=torch.bfloat16).to(DEV)
    gen = torch.Generator().manual_seed(78)
    O.reference_init_(list(stack.parameters()), gen)
    dense = torch.nn.Linear(2 * D, C).to(DEV)
    graph = E.build_graph(torch.from_numpy(batch.heads), torch.from_numpy(batch.sent_ptr), device=DEV)
    anchor = torch.from_numpy(batch.anchor).to(DEV)
    dist = E.tree_distance(graph, anchor)
    xp = torch.randn(batch.n_rows, D, generator=gen)
    targets = torch.arange(B) % C
    seen = _spy_fused_plan(monkeypatch)
    out, loss, dx = _run_stack(stack, dense, graph, xp.to(DEV), anchor, dist, targets)
    assert seen and seen[0] is not None and seen[0][0] == R          # the fused kernels ran, on rows_cap-row tiles
    sp = batch.sent_ptr
    sents = [(xp[sp[b]:sp[b + 1]], torch.from_numpy(O.dense_adjacency_from_heads(h, len(h))).float(),
              int(batch.anchor[b]), torch.tensor(O.tree_distance_bfs(h, int(batch.anchor[b]))))
             for b, h in enumerate(batch.heads_list())]
    ora = _oracle_run(stack, dense, sents, targets)
    tol = 2e-2
    assert rel(out.x_out, torch.cat(ora["x_out"])) < tol
    ora_g = _oracle_run(stack, dense, sents, targets, forced=_check_routing(out, ora, sp[:-1]))
    _compare(out, loss, dx, stack, dense, ora, ora_g, tol, Lyr)
    fused_logits, fused_x_out = out.logits.detach().clone(), out.x_out.detach().clone()
    # the unfused kernels (aggregate -> linear -> pool) on the same inputs
    monkeypatch.setattr(gated, "_FUSED", False)
    out_u, loss_u, dx_u = _run_stack(stack, dense, graph, xp.to(DEV), anchor, dist, targets)
    assert seen[-1] is None
    assert rel(out_u.logits, fused_logits) < tol and rel(out_u.x_out, fused_x_out) < tol
    ora_u = _oracle_run(stack, dense, sents, targets, forced=_check_routing(out_u, ora, sp[:-1]))
    _compare(out_u, loss_u, dx_u, stack, dense, ora, ora_u, tol, Lyr)


def test_dense_graph_over_512_entries_runs_unfused_and_matches_the_oracle(monkeypatch):
    """graph_from_dense accepts any symmetric 0/1 pattern.  A sentence with more than 512 CSR entries does not fit the
    fused kernels' tiles: the graph must report its largest sentence, tile_plan must refuse it, and the bf16 stack must
    still match the oracle (on the unfused kernels)."""
    import ed_gated_gcn_b200 as E
    from ed_gated_gcn_b200 import ops, synth
    from test_gpu_c_models import _check_routing, _compare, _oracle_run
    B, T, D, C, Lyr = 8, 48, 300, 34, 2
    rng = np.random.default_rng(48)
    adj = np.zeros((B, T, T), dtype=np.float32)
    for b in range(B):
        a = O.dense_adjacency_from_heads(synth.random_tree(T, rng), T).astype(np.float32)     # tree + identity
        extra = np.triu(rng.random((T, T)) < (0.35 if b == 3 else 0.05), 1)
        a[extra | extra.T] = 1.0
        adj[b] = a
    nnz = (adj != 0).sum((1, 2))
    assert nnz[3] > 512 and (np.delete(nnz, 3) <= 512).all()
    graph = E.graph_from_dense(torch.from_numpy(adj).to(DEV))
    assert graph.max_sent_nnz == int(nnz.max())
    assert graph.tile_plan(ops.fused_tile_rows(D, D)) is None
    torch.manual_seed(48)
    stack = E.GatedGCNStack(D, n_layers=Lyr, n_classes=C, gate_arch="sig-2", compute_dtype=torch.bfloat16).to(DEV)
    gen = torch.Generator().manual_seed(49)
    O.reference_init_(list(stack.parameters()), gen)
    dense = torch.nn.Linear(2 * D, C).to(DEV)
    xp = torch.randn(B * T, D, generator=gen)
    anchor = torch.from_numpy(rng.integers(0, T, B)).to(DEV)
    dist = E.tree_distance(graph, anchor)                     # the same distances go to both sides
    targets = torch.arange(B) % C
    seen = _spy_fused_plan(monkeypatch)
    out, loss, dx = _run_stack(stack, dense, graph, xp.to(DEV), anchor, dist, targets)
    assert seen == [None]
    dc = dist.cpu().long()
    sents = [(xp[b * T:(b + 1) * T], torch.from_numpy(adj[b]), int(anchor[b]), dc[b * T:(b + 1) * T]) for b in range(B)]
    ora = _oracle_run(stack, dense, sents, targets)
    ora_g = _oracle_run(stack, dense, sents, targets, forced=_check_routing(out, ora, [b * T for b in range(B)]))
    _compare(out, loss, dx, stack, dense, ora, ora_g, 2e-2, Lyr)
