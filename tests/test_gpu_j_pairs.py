"""Every candidate trigger of a sentence from one pass of the GCN chain (``GatedGCNStack.forward(..., pairs=)``).

The reference is the expanded batch: each sentence's rows repeated once per (sentence, trigger) pair, run through the
existing ``GatedGCNStack`` and through ``oracle.gated_block_ref`` (one call per pair).  ``dx`` of the grouped run is the
sum over a sentence's pairs of the oracle's per-pair input gradients, summed in fp64."""
import numpy as np
import pytest
import torch

from gpu_util import DEV, rel
from oracle import ref_oracle as O

pytestmark = pytest.mark.gpu


# ------------------------------------------------------------------------------------------------ layouts
def _lengths_batch(lengths, seed):
    from ed_gated_gcn_b200 import synth
    return synth.make_batch(len(lengths), 0, 0, seed=seed, lengths=np.asarray(lengths))


def _layout(name):
    """(TreeBatch, pair_ptr, anchor) of a named layout."""
    from ed_gated_gcn_b200 import synth
    if name == "mixed":
        # 0 pairs, 1 pair, every token a candidate, two pairs on one anchor, empty and 1-token sentences
        b = _lengths_batch([7, 0, 12, 1, 30, 5, 1, 0, 19, 3], seed=3)
        per = [[], [], [0, 3, 3, 11], [0], list(range(30)), [4], [], [], list(range(19)), [2, 2]]
    elif name == "windows":
        # lengths that straddle 72 KB row windows at D = 64 and runs of short sentences, every token a candidate
        L = [64, 65, 1, 1, 0, 127, 128, 2, 33, 31, 32, 96, 97, 0, 0]
        b = _lengths_batch(L, seed=4)
        per = [list(range(n)) for n in L]
    elif name == "long":
        # sentences longer than any row window next to short ones
        L = [300, 4, 129, 0, 200]
        b = _lengths_batch(L, seed=5)
        per = [[0, 150, 299, 150], [1, 2], list(range(0, 129, 3)), [], list(range(0, 200, 7))]
    elif name == "extra":
        b = synth.with_extra_edges(synth.make_batch(24, 1, 40, seed=9), rate=0.4, seed=10)
        pp, an = synth.candidate_pairs(b, per_sentence=3, none_rate=0.2, seed=11)
        return b, pp, an
    elif name == "512":
        b = _lengths_batch([512], seed=6)
        per = [list(range(512))]
    else:
        raise KeyError(name)
    pp = np.zeros(len(per) + 1, dtype=np.int32)
    pp[1:] = np.cumsum([len(p) for p in per])
    an = np.asarray([a for p in per for a in p], dtype=np.int32)
    return b, pp, an


def _dense_of(batch, s):
    from test_gpu_h_extra_edges import dense_of
    return dense_of(batch.heads_list()[s], batch.extras_list()[s])


def _graph(batch, **kw):
    import ed_gated_gcn_b200 as E
    if batch.extra_edges is not None:
        kw.update(extra_edges=torch.from_numpy(batch.extra_edges), edge_ptr=torch.from_numpy(batch.edge_ptr))
    return E.build_graph(torch.from_numpy(batch.heads), torch.from_numpy(batch.sent_ptr), device=DEV, **kw)


def _expand(batch, pp, an):
    """The expanded batch: sentence s copied once per pair.  Returns (TreeBatch, row index into the sentence rows)."""
    from ed_gated_gcn_b200 import synth
    sp = batch.sent_ptr
    owner = np.repeat(np.arange(batch.n_graphs), np.diff(pp))
    heads = [batch.heads[sp[s]:sp[s + 1]] for s in owner]
    lens = np.asarray([len(h) for h in heads], dtype=np.int32)
    esp = np.zeros(len(lens) + 1, dtype=np.int32)
    esp[1:] = np.cumsum(lens)
    rows = np.concatenate([np.arange(sp[s], sp[s + 1]) for s in owner] + [np.zeros(0, np.int64)])
    ex = ep = None
    if batch.extra_edges is not None:
        xl = [batch.extras_list()[s] for s in owner]
        ex = np.concatenate(xl + [np.zeros((0, 2), np.int32)]).astype(np.int32)
        ep = np.zeros(len(xl) + 1, dtype=np.int32)
        ep[1:] = np.cumsum([len(x) for x in xl])
    eb = synth.TreeBatch(heads=np.concatenate(heads + [np.zeros(0, np.int32)]).astype(np.int32), sent_ptr=esp,
                         anchor=an.astype(np.int32), lengths=lens, extra_edges=ex, edge_ptr=ep)
    return eb, torch.from_numpy(rows)


# ------------------------------------------------------------------------------------------------ runs
def _model(D, dtype, seed, Lyr=2, gated=True, gate_arch="sig-2", C=34):
    import ed_gated_gcn_b200 as E
    torch.manual_seed(seed)
    stack = E.GatedGCNStack(D, n_layers=Lyr, n_classes=C, gate_arch=gate_arch, compute_dtype=dtype, gated=gated).to(DEV)
    O.reference_init_(list(stack.parameters()), torch.Generator().manual_seed(seed + 1))
    dense = torch.nn.Linear(2 * D, C).to(DEV)
    return stack, dense


def _run(stack, dense, x0, graph, anchor, dist, targets, pairs=None):
    for p in list(stack.parameters()) + list(dense.parameters()):
        p.grad = None
    x = x0.clone().requires_grad_(True)
    out = stack(x, graph, anchor, dist, lambda a, p: dense(torch.cat([a, p], 1)), head_params=list(dense.parameters()),
                pairs=pairs)
    loss = torch.nn.functional.cross_entropy(out.logits, targets.to(DEV)) + 0.01 * out.xy + 0.01 * out.kl
    loss.backward()
    grads = {n: p.grad.detach().clone() for n, p in list(stack.named_parameters()) + [("dense.weight", dense.weight),
                                                                                   ("dense.bias", dense.bias)]
             if p.grad is not None}
    return out, loss.detach(), x.grad.detach(), grads


def _grouped(batch, pp, an, D, dtype, seed, **model_kw):
    """The grouped run and everything the references need."""
    import ed_gated_gcn_b200 as E
    stack, dense = _model(D, dtype, seed, **model_kw)
    graph = _graph(batch)
    pairs = E.pairs_from_ptr(graph, torch.from_numpy(pp), torch.from_numpy(an))
    anchor = torch.from_numpy(an).to(DEV)
    dist = E.tree_distance(graph, anchor, pairs=pairs)
    x = torch.randn(batch.n_rows, D, generator=torch.Generator().manual_seed(seed + 2))
    targets = torch.arange(len(an)) % dense.out_features
    res = _run(stack, dense, x.to(DEV), graph, anchor, dist, targets, pairs)
    return stack, dense, graph, pairs, anchor, dist, x, targets, res


def _sum_dx(dx_exp, rows, N):
    """Expanded-batch input gradients summed onto the sentence rows (fp64, in pair order)."""
    out = torch.zeros(N, dx_exp.shape[1], dtype=torch.float64)
    out.index_add_(0, rows, dx_exp.detach().double().cpu())
    return out


def _compare_expanded(res_g, res_e, rows, N, tol):
    out, loss, dx, grads = res_g
    oe, le, dxe, ge = res_e
    for k in ("logits", "pooled", "scores"):
        assert rel(getattr(out, k), getattr(oe, k)) < tol, k
    assert rel(out.xy, oe.xy) < tol and rel(out.kl, oe.kl) < tol and rel(loss, le) < tol
    assert rel(dx.double().cpu(), _sum_dx(dxe, rows, N)) < tol, "dx"
    for n, g in ge.items():
        if n == "fc.0.bias" or g.abs().max() < 1e-9:
            continue                       # c_b cancels inside the softmax: that gradient is rounding noise
        assert rel(grads[n], g) < tol, n


def _oracle(stack, dense, batch, pp, an, x, dist, targets, forced=None):
    from test_gpu_c_models import _oracle_run
    sp = batch.sent_ptr
    owner = np.repeat(np.arange(batch.n_graphs), np.diff(pp))
    dc = dist.cpu().long()
    sents, o = [], 0
    for p, s in enumerate(owner):
        n = int(sp[s + 1] - sp[s])
        sents.append((x[sp[s]:sp[s + 1]], torch.from_numpy(_dense_of(batch, s)).float(), int(an[p]), dc[o:o + n]))
        o += n
    ora = _oracle_run(stack, dense, sents, targets, forced=forced)
    return ora, owner


def _oracle_dx_per_sentence(ora, owner, batch):
    """The oracle's per-pair input gradients summed per sentence in fp64 (zeros for sentences without pairs)."""
    sp = batch.sent_ptr
    acc = [torch.zeros(int(sp[s + 1] - sp[s]), ora["dx"][0].shape[1] if ora["dx"] else 1, dtype=torch.float64)
           for s in range(batch.n_graphs)]
    for g, s in zip(ora["dx"], owner):
        acc[s] += g.double()
    return dict(ora, dx=acc)


# ------------------------------------------------------------------------------------------------ tests
@pytest.mark.parametrize("layout", ["mixed", "windows", "long", "extra"])
def test_fp32_pairs_vs_oracle_and_expanded(layout):
    """fp32: the grouped run against the per-pair oracle (dx summed per sentence) and against the existing stack on the
    expanded batch."""
    from test_gpu_c_models import _compare
    batch, pp, an = _layout(layout)
    D = 64
    stack, dense, graph, pairs, anchor, dist, x, targets, res = _grouped(batch, pp, an, D, torch.float32, 11)
    out, loss, dx, _ = res
    assert out.logits.shape == (len(an), 34) and out.scores.shape == (pairs.n_pair_rows,)
    assert out.pooled_arg.shape == (len(an), D) and out.view_arg.shape == (2, len(an), D)
    ora, owner = _oracle(stack, dense, batch, pp, an, x, dist, targets)
    _compare(out, loss, dx, stack, dense, ora, _oracle_dx_per_sentence(ora, owner, batch), 1e-5, 2)
    eb, rows = _expand(batch, pp, an)
    eg = _graph(eb)
    ea = torch.from_numpy(eb.anchor).to(DEV)
    res_e = _run(stack, dense, x[rows].to(DEV), eg, ea, _expand_dist(eg, ea), targets)
    assert torch.equal(_expand_dist(eg, ea), dist)                     # tree_distance(pairs=) = the expanded layout
    _compare_expanded(res, res_e, rows, batch.n_rows, 1e-4)


def _expand_dist(graph, anchor):
    import ed_gated_gcn_b200 as E
    return E.tree_distance(graph, anchor)


@pytest.mark.parametrize("fused", [True, False], ids=["fused", "unfused"])
@pytest.mark.parametrize("layout", ["mixed", "windows", "extra"])
def test_bf16_pairs_vs_oracle(layout, fused, monkeypatch):
    """bf16 on the fused plan and on the unfused kernels: forward against the oracle, gradients against the oracle run
    under this path's own max-pool routing (re-routed positions must be near-ties)."""
    from ed_gated_gcn_b200 import gated
    from test_gpu_c_models import _check_routing, _compare
    from test_gpu_g_fused_limits import _spy_fused_plan
    monkeypatch.setattr(gated, "_FUSED", fused)
    seen = _spy_fused_plan(monkeypatch)
    batch, pp, an = _layout(layout)
    D = 64
    stack, dense, graph, pairs, anchor, dist, x, targets, res = _grouped(batch, pp, an, D, torch.bfloat16, 21)
    assert (seen[0] is not None) == fused
    out, loss, dx, _ = res
    ora, owner = _oracle(stack, dense, batch, pp, an, x, dist, targets)
    starts = torch.from_numpy(batch.sent_ptr[:-1][owner].astype(np.int64))
    ora_g, _ = _oracle(stack, dense, batch, pp, an, x, dist, targets, forced=_check_routing(out, ora, starts))
    _compare(out, loss, dx, stack, dense, ora, _oracle_dx_per_sentence(ora_g, owner, batch), 2e-2, 2)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
@pytest.mark.parametrize("variant", ["ungated", "L3", "gate-2", "gate-3", "gate-sig-3"])
def test_pairs_model_variants_vs_expanded(variant, dtype):
    """gated=False, L = 3 and every gate architecture against the existing stack on the expanded batch (fp32), and
    against the oracle under this path's routing (bf16)."""
    from test_gpu_c_models import _check_routing, _compare
    kw = dict(ungated=dict(gated=False), L3=dict(Lyr=3), **{"gate-2": dict(gate_arch="2"), "gate-3": dict(gate_arch="3"),
                                                            "gate-sig-3": dict(gate_arch="sig-3")})[variant]
    batch, pp, an = _layout("mixed")
    D = 64
    stack, dense, graph, pairs, anchor, dist, x, targets, res = _grouped(batch, pp, an, D, dtype, 31, **kw)
    Lyr = kw.get("Lyr", 2)
    out, loss, dx, _ = res
    if dtype == torch.float32:
        eb, rows = _expand(batch, pp, an)
        eg = _graph(eb)
        ea = torch.from_numpy(eb.anchor).to(DEV)
        res_e = _run(stack, dense, x[rows].to(DEV), eg, ea, _expand_dist(eg, ea), targets)
        _compare_expanded(res, res_e, rows, batch.n_rows, 1e-4)
        return
    if not kw.get("gated", True):
        return                              # the oracle helper runs the gated block
    ora, owner = _oracle(stack, dense, batch, pp, an, x, dist, targets)
    starts = torch.from_numpy(batch.sent_ptr[:-1][owner].astype(np.int64))
    ora_g, _ = _oracle(stack, dense, batch, pp, an, x, dist, targets, forced=_check_routing(out, ora, starts))
    _compare(out, loss, dx, stack, dense, ora, _oracle_dx_per_sentence(ora_g, owner, batch), 2e-2, Lyr)


def test_512_token_sentence_with_512_pairs_vs_expanded():
    batch, pp, an = _layout("512")
    D = 64
    stack, dense, graph, pairs, anchor, dist, x, targets, res = _grouped(batch, pp, an, D, torch.float32, 41)
    eb, rows = _expand(batch, pp, an)
    eg = _graph(eb)
    ea = torch.from_numpy(eb.anchor).to(DEV)
    res_e = _run(stack, dense, x[rows].to(DEV), eg, ea, _expand_dist(eg, ea), targets)
    _compare_expanded(res, res_e, rows, batch.n_rows, 1e-4)


@pytest.mark.parametrize("layout", ["mixed", "long", "extra", "512"])
def test_tree_distance_pairs_bit_exact(layout):
    """tree_distance(pairs=) against a per-pair breadth-first search of the sentence's pattern."""
    import ed_gated_gcn_b200 as E
    from test_gpu_h_extra_edges import tree_dist_bfs
    batch, pp, an = _layout(layout)
    graph = _graph(batch)
    pairs = E.pairs_from_ptr(graph, torch.from_numpy(pp), torch.from_numpy(an))
    got = E.tree_distance(graph, torch.from_numpy(an).to(DEV), pairs=pairs).cpu().numpy()
    owner = np.repeat(np.arange(batch.n_graphs), np.diff(pp))
    want = [tree_dist_bfs(_dense_of(batch, s), int(a)) for s, a in zip(owner, an)]
    want = np.concatenate(want + [np.zeros(0, np.int64)])
    assert np.array_equal(got, want)
    if batch.extra_edges is None:
        for p, (s, a) in enumerate(zip(owner, an)):
            o = int(pairs.pair_row_ptr[p])
            h = batch.heads_list()[s]
            assert got[o:o + len(h)].tolist() == O.tree_distance_bfs(h, int(a))


def test_two_runs_are_bitwise_equal():
    batch, pp, an = _layout("windows")
    for dtype in (torch.bfloat16, torch.float32):
        r1 = _grouped(batch, pp, an, 64, dtype, 51)[-1]
        r2 = _grouped(batch, pp, an, 64, dtype, 51)[-1]
        for k in ("logits", "xy", "kl", "scores", "pooled", "pooled_arg", "view_arg"):
            assert torch.equal(getattr(r1[0], k), getattr(r2[0], k)), k
        assert torch.equal(r1[2], r2[2])
        for n in r1[3]:
            assert torch.equal(r1[3][n], r2[3][n]), n


def test_captured_step_without_host_sync():
    """graph build (max_len given), pairs_from_ptr (n_pair_rows given), tree_distance(pairs=) and the training step in
    one CUDA graph (a device->host read during capture raises); the replay gives the eager result."""
    import ed_gated_gcn_b200 as E
    from ed_gated_gcn_b200 import synth
    from ed_gated_gcn_b200.runtime import GraphedStep
    batch = synth.config_batch("C2", n_graphs=96)
    pp, an = synth.candidate_pairs(batch)
    D = 300
    stack, _ = _model(D, torch.bfloat16, 61)
    head = E.DenseHead(2 * D, 34).to(DEV)
    st = dict(h=torch.from_numpy(batch.heads).to(DEV), sp=torch.from_numpy(batch.sent_ptr).to(DEV),
              pp=torch.from_numpy(pp).to(DEV), an=torch.from_numpy(an).to(DEV),
              tg=(torch.arange(len(an)) % 34).to(DEV))
    x = torch.randn(batch.n_rows, D, generator=torch.Generator().manual_seed(62)).to(DEV).requires_grad_(True)
    max_len, n_pair_rows = int(batch.lengths.max()), int((batch.lengths.astype(np.int64) ** 2).sum())
    res = {}

    def step():
        for p in list(stack.parameters()) + list(head.parameters()):
            p.grad = None
        x.grad = None
        g = E.build_graph(st["h"], st["sp"], max_len=max_len)
        pairs = E.pairs_from_ptr(g, st["pp"], st["an"], n_pair_rows=n_pair_rows)
        d = E.tree_distance(g, st["an"], pairs=pairs)
        out = stack(x, g, st["an"], d, head, pairs=pairs)
        loss = E.total_loss(E.cross_entropy(out.logits, st["tg"]), out.xy, out.kl, 0.01, 0.01)
        loss.backward()
        res.update(loss=loss.detach(), logits=out.logits.detach(), scores=out.scores.detach(), dx=x.grad,
                   gw=stack.gc1.weight.grad)
        return loss

    step()
    eager = {k: v.clone() for k, v in res.items()}
    gs = GraphedStep(step)
    gs()
    torch.cuda.synchronize()
    for k, v in eager.items():
        assert torch.equal(res[k], v), k


def test_declined_combinations_raise():
    import ed_gated_gcn_b200 as E
    batch, pp, an = _layout("mixed")
    D = 64
    graph = _graph(batch)
    pairs = E.pairs_from_ptr(graph, torch.from_numpy(pp), torch.from_numpy(an))
    anchor = torch.from_numpy(an).to(DEV)
    dist = E.tree_distance(graph, anchor, pairs=pairs)
    x = torch.randn(batch.n_rows, D, device=DEV)
    dense = torch.nn.Linear(2 * D, 2).to(DEV)                  # as many classes as the stacks' fc (n_classes=2)
    fn = lambda a, p: dense(torch.cat([a, p], 1))

    def call(stack, **kw):
        with pytest.raises(E.EdgError, match=kw.pop("match")):
            stack(kw.pop("x", x), graph, anchor, dist, fn, head_params=list(dense.parameters()), pairs=pairs, **kw)

    s = E.GatedGCNStack(D, dropout=0.3, compute_dtype=torch.bfloat16).to(DEV).train()
    call(s, match="gate dropout")
    s.eval()
    s(x, graph, anchor, dist, fn, head_params=list(dense.parameters()), pairs=pairs)     # eval mode: dropout is off
    wide = torch.nn.Linear(2 * D, 34).to(DEV)                  # more classes than the fc head scores
    with pytest.raises(E.EdgError, match="classes"):
        s(x, graph, anchor, dist, lambda a, p: wide(torch.cat([a, p], 1)), head_params=list(wide.parameters()),
          pairs=pairs)
    call(E.GatedGCNStack(D, fc_sigmoid=True).to(DEV), match="fc_sigmoid")
    base = E.GatedGCNStack(D).to(DEV)
    call(base, match="view_len", view_len=torch.ones(batch.n_graphs, dtype=torch.int64, device=DEV))
    call(base, match="aspect", aspect=torch.zeros(len(an), D, device=DEV))
    call(base, match="return_x_out", return_x_out=True)
    call(base, match="3-D", x=x[None])
    with pytest.raises(E.EdgError, match="per-pair packed"):
        base(x, graph, anchor, dist[:-1], fn, head_params=list(dense.parameters()), pairs=pairs)
    with pytest.raises(E.EdgError, match="tree_distance"):
        E.tree_distance(graph, anchor, pad="zero", pairs=pairs)
