"""The fused layer kernel (edg_gcn_layer: projection + tree aggregation + max-pool in one launch) through the
C ABI, against fp64 CPU torch built from the oracle's dense adjacency (models/gcn.py:33-45 in the reference's own
association  adj @ (x @ W) / denom + b), and against the unfused kernels on the same inputs.  bf16: <= 2e-2."""
import numpy as np
import pytest
import torch

from gpu_util import DEV, rel
from oracle import ref_oracle as O

pytestmark = pytest.mark.gpu


def _setup(B, lo, hi, seed, D, Nout):
    import ed_gated_gcn_b200 as E
    from ed_gated_gcn_b200 import ops, synth
    batch = synth.make_batch(B, lo, hi, seed=seed)
    g = E.build_graph(torch.from_numpy(batch.heads), torch.from_numpy(batch.sent_ptr), device=DEV)
    gen = torch.Generator().manual_seed(seed)
    x = torch.randn(batch.n_rows, D, generator=gen)
    w = torch.randn(Nout, D, generator=gen) / D ** 0.5
    bias = torch.randn(Nout, generator=gen)
    xr, wr = ops.as_rows(x.to(DEV), torch.bfloat16), ops.as_rows(w.to(DEV), torch.bfloat16)
    rows = ops.fused_tile_rows(D, Nout)
    assert rows >= 32
    plan = g.tile_plan(rows)
    assert plan is not None
    return batch, g, xr, wr, bias, rows, plan


def _dense_ops(batch):
    """per sentence: A^ = A / (rowsum + 1) as fp64 (gcn.py:35, 41)"""
    out = []
    for h in batch.heads_list():
        a = torch.from_numpy(O.dense_adjacency_from_heads(h, len(h))).double()
        out.append(a / (a.sum(1, keepdim=True) + 1))
    return out


def check_tile_plan(sp, g, rows, plan):
    """The tiles of edg_tile_plan cover every sentence once, in order, greedily, within the row, sentence and CSR-entry
    caps of the fused kernels; returns the plan's tile_info rows on the host."""
    from ed_gated_gcn_b200 import ops
    info, n_tiles = plan
    nt = int(n_tiles.item())
    info = info[:nt].cpu().numpy()
    rp = g.row_ptr.cpu().numpy()
    assert info[0, 0] == 0 and info[-1, 1] == len(sp) - 1
    assert np.array_equal(info[1:, 0], info[:-1, 1])
    assert np.array_equal(info[:, 2], sp[info[:, 0]]) and np.array_equal(info[:, 3], sp[info[:, 1]])
    assert np.array_equal(info[:, 4], rp[info[:, 2]]) and np.array_equal(info[:, 5], rp[info[:, 3]])
    assert ((info[:, 3] - info[:, 2]) <= rows).all() and ((info[:, 1] - info[:, 0]) <= ops.FUSED_MAX_SENTENCES).all()
    assert ((info[:, 5] - info[:, 4]) <= 512).all()
    assert ((info[:, 1] - info[:, 0]) >= 1).all()
    # greedy: the next sentence would not have fitted (rows or CSR entries) unless the sentence cap stopped the tile
    for t in range(nt - 1):
        s1 = info[t, 1]
        full = (sp[s1 + 1] - info[t, 2] > rows) or (rp[sp[s1 + 1]] - info[t, 4] > 512) \
            or (info[t, 1] - info[t, 0] == ops.FUSED_MAX_SENTENCES)
        assert full, t
    return info


def test_tile_plan_covers_every_sentence_once():
    batch, g, _, _, _, rows, plan = _setup(700, 1, 50, 3, 64, 64)
    check_tile_plan(batch.sent_ptr, g, rows, plan)


@pytest.mark.parametrize("shape", [(300, 300), (64, 64), (256, 256), (300, 160), (128, 320), (48, 16)])
def test_fused_forward_layer_and_pool(shape):
    from ed_gated_gcn_b200 import ops
    D, Nout = shape
    batch, g, xr, wr, bias, rows, plan = _setup(157, 1, 50, 11 + D, D, Nout)
    y, hmax, harg, _ = ops.gcn_layer(xr, wr, bias.to(DEV), g, 0, plan, rows, want_pool=True)
    xd, wd = xr.float().cpu().double(), wr.float().cpu().double()
    want = []
    for b, ah in enumerate(_dense_ops(batch)):
        lo, hi = batch.sent_ptr[b], batch.sent_ptr[b + 1]
        want.append(ah @ (xd[lo:hi] @ wd.t()) + bias.double())
    want = torch.cat(want)
    assert rel(y.float(), want) < 8e-3
    base = y.as_strided((y.shape[0], y.stride(0)), (y.stride(0), 1))
    assert torch.isfinite(base.float()).all() and (base[:, Nout:] == 0).all()
    # the pool is the exact column maximum of the STORED bf16 rows, first row on ties (torch.max semantics)
    yc = y.float().cpu()
    for b in range(batch.n_graphs):
        lo, hi = int(batch.sent_ptr[b]), int(batch.sent_ptr[b + 1])
        m, a = yc[lo:hi].max(0)
        assert torch.equal(hmax[b].cpu(), m), b
        # first index of the maximum
        first = (yc[lo:hi] == m[None]).float().argmax(0) + lo
        assert torch.equal(harg[b].cpu().long(), first), b
    # against the unfused kernels (aggregate -> linear): same operation in the other association
    y2 = ops.linear(ops.aggregate(xr, g, mode=0), wr, bias.to(DEV))
    assert rel(y.float(), y2.float()) < 1.5e-2


@pytest.mark.parametrize("shape", [(300, 300), (64, 64), (300, 160)])
def test_fused_adjoint_layer_patch_and_colsum(shape):
    from ed_gated_gcn_b200 import ops
    D, Nout = shape
    batch, g, xr, wr, _, rows, plan = _setup(143, 1, 50, 5 + D, D, Nout)
    B = batch.n_graphs
    gen = torch.Generator().manual_seed(1)
    pv = torch.randn(B, Nout, generator=gen)
    # one arg row per (sentence, column), some entries switched off
    lens = torch.from_numpy(batch.lengths.astype(np.int64))
    starts = torch.from_numpy(batch.sent_ptr[:-1].astype(np.int64))
    pa = (torch.rand(B, Nout, generator=gen) * lens[:, None]).long().clamp_max((lens - 1).clamp_min(0)[:, None]) + starts[:, None]
    pa[torch.rand(B, Nout, generator=gen) < 0.2] = -1
    pa[lens == 0] = -1
    xd, wd = xr.float().cpu().double(), wr.float().cpu().double()
    u = xd @ wd.t()
    patched = u.clone()
    bi, ci = torch.nonzero(pa >= 0, as_tuple=True)
    patched[pa[bi, ci], ci] += pv[bi, ci].double()
    want, want_plain = [], []
    for b, ah in enumerate(_dense_ops(batch)):
        lo, hi = batch.sent_ptr[b], batch.sent_ptr[b + 1]
        want.append(ah.t() @ patched[lo:hi])
        want_plain.append(ah.t() @ u[lo:hi])
    want, want_plain = torch.cat(want), torch.cat(want_plain)
    y, _, _, cs = ops.gcn_layer(xr, wr, None, g, 1, plan, rows, patch=(pv.to(DEV), pa.int().to(DEV)), want_colsum=True)
    assert rel(y.float(), want) < 8e-3
    # the column sums ride along the gather of the bf16-staged rows (as the unfused path's came from bf16 dh)
    assert rel(cs, patched.sum(0)) < 5e-3
    y0, _, _, cs0 = ops.gcn_layer(xr, wr, None, g, 1, plan, rows, want_colsum=True)
    assert rel(y0.float(), want_plain) < 8e-3
    assert rel(cs0, u.sum(0)) < 5e-3
    y1 = ops.aggregate(ops.linear(xr, wr, None), g, mode=1)
    assert rel(y0.float(), y1.float()) < 1.5e-2


def test_fused_layer_config2_size_invariants():
    """C2-sized batch (4096 trees): deterministic across launches, and equal to the small-batch result sentence
    by sentence (tiles are independent)."""
    from ed_gated_gcn_b200 import ops, synth
    import ed_gated_gcn_b200 as E
    batch = synth.config_batch("C2")
    g = E.build_graph(torch.from_numpy(batch.heads), torch.from_numpy(batch.sent_ptr), device=DEV)
    D = 300
    gen = torch.Generator().manual_seed(0)
    x = torch.randn(batch.n_rows, D, generator=gen)
    w = torch.randn(D, D, generator=gen) / D ** 0.5
    bias = torch.randn(D, generator=gen)
    xr, wr = ops.as_rows(x.to(DEV), torch.bfloat16), ops.as_rows(w.to(DEV), torch.bfloat16)
    rows = ops.fused_tile_rows(D, D)
    plan = g.tile_plan(rows)
    y, hmax, harg, _ = ops.gcn_layer(xr, wr, bias.to(DEV), g, 0, plan, rows, want_pool=True)
    y_again, hmax2, harg2, _ = ops.gcn_layer(xr, wr, bias.to(DEV), g, 0, plan, rows, want_pool=True)
    assert torch.equal(y, y_again) and torch.equal(hmax, hmax2) and torch.equal(harg, harg2)
    # a 64-sentence sample against fp64
    xd, wd = xr.float().cpu().double(), wr.float().cpu().double()
    yc = y.float().cpu()
    heads = batch.heads_list()
    for b in range(0, batch.n_graphs, 64):
        lo, hi = int(batch.sent_ptr[b]), int(batch.sent_ptr[b + 1])
        a = torch.from_numpy(O.dense_adjacency_from_heads(heads[b], hi - lo)).double()
        want = (a / (a.sum(1, keepdim=True) + 1)) @ (xd[lo:hi] @ wd.t()) + bias.double()
        assert rel(yc[lo:hi], want) < 8e-3, b
        assert torch.equal(hmax[b].cpu(), yc[lo:hi].max(0)[0]), b
    # pool against the stand-alone pool kernel with a unit gate
    ones = torch.ones((1, batch.n_graphs, D), dtype=torch.float32, device=DEV)
    pooled, arg = ops.pool_fwd(y, g, ones)
    assert torch.equal(pooled[0], hmax) and torch.equal(arg[0], harg)


@pytest.mark.parametrize("with_scores_grad", [False, True])
@pytest.mark.parametrize("D", [300, 64])
def test_head_du_matches_head_bwd_then_aggregate(D, with_scores_grad):
    """edg_head_du (top-layer gradient generated in aggregated form from row scalars and sentence vectors) against the
    kernels it replaces: edg_head_bwd (dh_L, d gate_L) -> edg_aggregate mode 1, edg_colsum."""
    import ed_gated_gcn_b200 as E
    from ed_gated_gcn_b200 import ops, synth
    batch = synth.make_batch(211, 1, 50, seed=7 + D)
    g = E.build_graph(torch.from_numpy(batch.heads), torch.from_numpy(batch.sent_ptr), device=DEV)
    B, N = batch.n_graphs, batch.n_rows
    gen = torch.Generator().manual_seed(3)
    h = ops.as_rows(torch.randn(N, D, generator=gen).to(DEV), torch.bfloat16)
    gate = torch.rand(B, D, generator=gen).to(DEV) * 0.9 + 0.05
    v = (torch.randn(B, D, generator=gen) * 0.2).to(DEV)
    c = torch.randn(B, generator=gen).to(DEV)
    gp = torch.randn(B, D, generator=gen).to(DEV)
    anchor = torch.from_numpy(batch.anchor).to(DEV)
    dist = E.tree_distance(g, anchor)
    rows = ops.fused_tile_rows(D, D)
    plan = g.tile_plan(rows)
    scores, kl_b, kl, dvu, dcu, uu, sfu = ops.scores_kl_fwd(h, g, gate, v, c, dist, want_units=True, want_rows=True)
    ones = torch.ones((1, B, D), dtype=torch.float32, device=DEV)
    hmax_all, arg_all = ops.pool_fwd(h, g, ones)
    hmax, arg = hmax_all[0].contiguous(), arg_all[0].contiguous()
    g_kl = torch.tensor(0.37, device=DEV)
    g_sc = (torch.randn(N, generator=gen) * 0.1).to(DEV) if with_scores_grad else None
    dh, dgate_ref, _, _ = ops.head_bwd(h, g, gate, v, dist, scores, kl_b, g_kl, g_sc, gp, arg, None, want_dh=True, want_dv=False)
    want_du = ops.aggregate(dh, g, mode=1, out_dtype=torch.float32)
    want_db = dh.float().sum(0)
    du, db, dgate = ops.head_du(uu, g_kl, g_sc, gate, v, gp, arg, sfu, hmax, g, plan)
    # dh_L itself is rounded to bf16 on the reference side before it is aggregated; head_du rounds once at the end
    assert rel(du.float(), want_du) < 8e-3
    assert rel(db, want_db) < 5e-3
    base = du.as_strided((N, du.stride(0)), (du.stride(0), 1))
    assert torch.isfinite(base.float()).all() and (base[:, D:] == 0).all()
    if not with_scores_grad:                 # (with a gradient on scores the caller adds sum_t g_scores_t h_t itself)
        assert rel(dgate, dgate_ref) < 1e-4
    # fp64 check of du on a few sentences from the definition
    ds = (g_kl.double().cpu() * uu.double().cpu()) + (g_sc.double().cpu() if g_sc is not None else 0)
    for b in range(0, B, 37):
        lo, hi = int(batch.sent_ptr[b]), int(batch.sent_ptr[b + 1])
        if hi == lo:
            continue
        a = torch.from_numpy(O.dense_adjacency_from_heads(batch.heads_list()[b], hi - lo)).double()
        ah = a / (a.sum(1, keepdim=True) + 1)
        q = (gate[b] * v[b]).double().cpu()
        dh64 = ds[lo:hi, None] * q[None]
        ar = arg[b].cpu().long() - lo
        dh64[ar, torch.arange(D)] += (gate[b] * gp[b]).double().cpu()
        assert rel(du[lo:hi].float(), ah.t() @ dh64) < 8e-3, b


def test_bucket_hook_backward_equals_plain_backward():
    """`GatedGCNStack.grad_bucket_hook` (what parallel.GradientAllReducer.bucket plugs into): the backward pass hands all
    parameter gradients over before the input-gradient projection, gets views of one flat buffer back and runs that
    projection on fewer SMs.  With a hook that only packs, every gradient must equal the plain pass bit for bit, and
    every parameter's .grad must live inside the flat buffer."""
    import ed_gated_gcn_b200 as E
    from ed_gated_gcn_b200 import synth
    torch.manual_seed(7)
    D, C, B = 300, 34, 600
    batch = synth.make_batch(B, 5, 50, seed=11)
    stack = E.GatedGCNStack(D, n_layers=2, n_classes=C, gate_arch="sig-2", compute_dtype=torch.bfloat16).to(DEV)
    dense = torch.nn.Linear(2 * D, C).to(DEV)
    graph = E.build_graph(torch.from_numpy(batch.heads), torch.from_numpy(batch.sent_ptr), device=DEV)
    anchor = torch.from_numpy(batch.anchor).to(DEV)
    dist = E.tree_distance(graph, anchor)
    x = torch.randn(batch.n_rows, D, device=DEV).requires_grad_(True)
    tgt = (torch.arange(B) % C).to(DEV)
    params = list(stack.parameters()) + list(dense.parameters())

    def run():
        for p in params:
            p.grad = None
        x.grad = None
        out = stack(x, graph, anchor, dist, lambda a, p: dense(torch.cat([a, p], 1)), head_params=list(dense.parameters()))
        (torch.nn.functional.cross_entropy(out.logits, tgt) + 0.01 * out.xy + 0.01 * out.kl).backward()
        return [p.grad for p in params], x.grad

    g_plain, dx_plain = run()
    seen = {}

    def pack_only(tensors):
        idx = [i for i, t in enumerate(tensors) if t is not None and t.dtype == torch.float32]
        flat = torch.cat([tensors[i].reshape(-1) for i in idx])
        seen["flat"], seen["n"] = flat, len(idx)
        out, off = list(tensors), 0
        for i in idx:
            out[i] = flat[off:off + tensors[i].numel()].view_as(tensors[i])
            off += tensors[i].numel()
        return out

    stack.grad_bucket_hook = pack_only
    g_hook, dx_hook = run()
    assert seen["n"] == len(params)
    assert torch.equal(dx_hook, dx_plain)
    lo, hi = seen["flat"].data_ptr(), seen["flat"].data_ptr() + seen["flat"].numel() * 4
    for a, b in zip(g_hook, g_plain):
        assert torch.equal(a, b)
        assert lo <= a.data_ptr() < hi          # autograd installed the view itself: nothing was copied back
