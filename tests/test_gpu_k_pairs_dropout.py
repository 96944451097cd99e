"""Train-mode gate dropout on grouped trigger pairs (``GatedGCNStack(dropout=p, pair_dropout=True)``, ``pairs=``).

Pair p applies the masks the expanded batch applies to its copy of the sentence (``edg_dropout_rows`` keyed on the
per-pair packed row ``pair_row_ptr[p] + t``), so for one seed the grouped run reproduces the existing stack on the
expanded batch -- the arg-max rows exactly -- and the oracle run per pair with the same masks rebuilt with numpy."""
import numpy as np
import pytest
import torch

from gpu_util import DEV, rel
from oracle import ref_oracle as O
from test_gpu_c_models import _compare, _dropout_mask_numpy, _oracle_params
from test_gpu_j_pairs import (_compare_expanded, _dense_of, _expand, _expand_dist, _graph, _layout,
                              _oracle_dx_per_sentence, _run)

pytestmark = pytest.mark.gpu

P_DROP = 0.25


def _model(D, dtype, seed, Lyr=2, p=P_DROP, gated=True, pair_dropout=True, C=34):
    import ed_gated_gcn_b200 as E
    torch.manual_seed(seed)
    stack = E.GatedGCNStack(D, n_layers=Lyr, n_classes=C, compute_dtype=dtype, gated=gated, dropout=p,
                            pair_dropout=pair_dropout).to(DEV).train()
    O.reference_init_(list(stack.parameters()), torch.Generator().manual_seed(seed + 1))
    dense = torch.nn.Linear(2 * D, C).to(DEV)
    return stack, dense


def _inputs(batch, pp, an, D, seed):
    import ed_gated_gcn_b200 as E
    graph = _graph(batch)
    pairs = E.pairs_from_ptr(graph, torch.from_numpy(pp), torch.from_numpy(an))
    anchor = torch.from_numpy(an).to(DEV)
    dist = E.tree_distance(graph, anchor, pairs=pairs)
    x = torch.randn(batch.n_rows, D, generator=torch.Generator().manual_seed(seed + 2))
    targets = torch.arange(len(an)) % 34
    return graph, pairs, anchor, dist, x, targets


def _grouped_and_expanded(layout, D, dtype, Lyr, seed):
    batch, pp, an = _layout(layout)
    stack, dense = _model(D, dtype, seed, Lyr=Lyr)
    graph, pairs, anchor, dist, x, targets = _inputs(batch, pp, an, D, seed)
    torch.manual_seed(seed + 3)
    res_g = _run(stack, dense, x.to(DEV), graph, anchor, dist, targets, pairs)
    seed_g = int(stack.last_dropout_seed)
    eb, rows = _expand(batch, pp, an)
    eg = _graph(eb)
    ea = torch.from_numpy(eb.anchor).to(DEV)
    torch.manual_seed(seed + 3)
    res_e = _run(stack, dense, x[rows].to(DEV), eg, ea, _expand_dist(eg, ea), targets)
    seed_e = int(stack.last_dropout_seed)
    return batch, pairs, rows, res_g, res_e, seed_g, seed_e


def _to_sentence_rows(arg, rows):
    """expanded-batch rows -> sentence rows (-1 stays -1)."""
    a = arg.cpu().long()
    return torch.where(a >= 0, rows[a.clamp_min(0)], a)


def _check_args_equal(out_g, out_e, rows):
    assert torch.equal(out_g.pooled_arg.cpu().long(), _to_sentence_rows(out_e.pooled_arg, rows)), "pooled_arg"
    assert torch.equal(out_g.view_arg.cpu().long(), _to_sentence_rows(out_e.view_arg, rows)), "view_arg"


@pytest.mark.parametrize("Lyr", [2, 3])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
@pytest.mark.parametrize("layout", ["mixed", "windows", "long", "extra"])
def test_dropout_pairs_vs_expanded_same_seed(layout, dtype, Lyr, monkeypatch):
    """Same torch seed before each arm: same dropout seed, the same masks, the same arg-max rows and (within the
    expanded comparison's tolerances) the same outputs and gradients."""
    if dtype == torch.float32:
        # the expanded batch crosses the row count above which fp32 projections run in split tensor-core form, the
        # sentences do not: on one projection kernel both arms compute bit-identical rows, so equal masks must give
        # equal arg-max rows (with two kernels, near-ties could legitimately flip)
        monkeypatch.setenv("EDG_F32_TC", "0")
    batch, pairs, rows, res_g, res_e, seed_g, seed_e = _grouped_and_expanded(layout, 64, dtype, Lyr, 71 + Lyr)
    assert seed_g == seed_e
    _check_args_equal(res_g[0], res_e[0], rows)
    _compare_expanded(res_g, res_e, rows, batch.n_rows, 1e-4 if dtype == torch.float32 else 2e-2)


def _oracle_drop(stack, dense, batch, pp, an, x, dist, targets, seed, n_pair_rows):
    """``gated_block_ref`` once per pair with the pair's masks (numpy, at its per-pair packed rows)."""
    sd, dw, db, gcn_p, gate_p, lead = _oracle_params(stack, dense)
    D, Lyr = x.shape[1], stack.n_layers
    masks = [torch.from_numpy(_dropout_mask_numpy(seed, v, P_DROP, n_pair_rows, D)) for v in range(Lyr)]
    sp = batch.sent_ptr
    owner = np.repeat(np.arange(batch.n_graphs), np.diff(pp))
    dc = dist.cpu().long()
    P = len(an)
    xs, logits, scores = [], [], []
    xy = kl = 0.0
    o = 0
    for p, s in enumerate(owner):
        lo, hi = int(sp[s]), int(sp[s + 1])
        n = hi - lo
        xb = x[lo:hi].clone().requires_grad_(True)
        adj = torch.from_numpy(_dense_of(batch, s)).float()
        r = O.gated_block_ref(xb[None], adj[None], torch.tensor([int(an[p])]), dc[o:o + n][None], gcn_p, gate_p,
                              sd["fc.0.weight"], sd["fc.0.bias"], lambda a, q: torch.cat([a, q], 1) @ dw.t() + db,
                              lead_sigmoid=lead, gate_masks=[m[o:o + n][None] for m in masks])
        xs.append(xb); logits.append(r["logits"]); scores.append(r["scores"][0])
        xy = xy + r["xy"] / P
        kl = kl + r["kl"] / P
        o += n
    lg = torch.cat(logits)
    loss = torch.nn.functional.cross_entropy(lg, targets) + 0.01 * xy + 0.01 * kl
    loss.backward()
    grads = {k: v.grad for k, v in sd.items()}
    grads["dense.weight"], grads["dense.bias"] = dw.grad, db.grad
    ora = dict(logits=lg, scores=scores, xy=xy, kl=kl, loss=loss, dx=[t.grad for t in xs], grads=grads)
    return ora, owner, masks


@pytest.mark.parametrize("layout", ["mixed", "extra"])
def test_dropout_pairs_vs_oracle_f32(layout):
    batch, pp, an = _layout(layout)
    D = 64
    stack, dense = _model(D, torch.float32, 81)
    graph, pairs, anchor, dist, x, targets = _inputs(batch, pp, an, D, 81)
    out, loss, dx, _ = _run(stack, dense, x.to(DEV), graph, anchor, dist, targets, pairs)
    ora, owner, masks = _oracle_drop(stack, dense, batch, pp, an, x, dist, targets, int(stack.last_dropout_seed),
                                     pairs.n_pair_rows)
    assert 0.68 < float((masks[0] > 0).float().mean()) < 0.82
    _compare(out, loss, dx, stack, dense, ora, _oracle_dx_per_sentence(ora, owner, batch), 1e-5, stack.n_layers)


def test_pairs_of_one_sentence_draw_independent_masks():
    """Every token a candidate: the view arg-max rows of the pairs of one sentence differ in some columns (a mask keyed
    on the sentence row would give every pair of the sentence the same rows)."""
    batch, pp, an = _layout("windows")
    D = 64
    stack, dense = _model(D, torch.float32, 91)
    graph, pairs, anchor, dist, x, targets = _inputs(batch, pp, an, D, 91)
    out = _run(stack, dense, x.to(DEV), graph, anchor, dist, targets, pairs)[0]
    va = out.view_arg.cpu()
    checked = 0
    for s in range(batch.n_graphs):
        p0, p1 = int(pp[s]), int(pp[s + 1])
        if p1 - p0 < 2 or batch.sent_ptr[s + 1] - batch.sent_ptr[s] < 8:
            continue
        for v in range(va.shape[0]):
            assert (va[v, p0] != va[v, p0 + 1]).any(), (s, v)
        checked += 1
    assert checked > 5


def test_512_token_sentence_with_512_pairs_vs_expanded_bf16():
    batch, pairs, rows, res_g, res_e, seed_g, seed_e = _grouped_and_expanded("512", 64, torch.bfloat16, 2, 101)
    assert seed_g == seed_e
    _check_args_equal(res_g[0], res_e[0], rows)
    _compare_expanded(res_g, res_e, rows, batch.n_rows, 2e-2)


def _bitwise_equal(r1, r2):
    for k in ("logits", "xy", "kl", "scores", "pooled", "pooled_arg", "view_arg"):
        assert torch.equal(getattr(r1[0], k), getattr(r2[0], k)), k
    assert torch.equal(r1[1], r2[1]) and torch.equal(r1[2], r2[2])
    assert r1[3].keys() == r2[3].keys()
    for n in r1[3]:
        assert torch.equal(r1[3][n], r2[3][n]), n


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
def test_no_op_cases(dtype):
    import ed_gated_gcn_b200 as E
    batch, pp, an = _layout("mixed")
    D = 64
    graph, pairs, anchor, dist, x, targets = _inputs(batch, pp, an, D, 111)
    xd = x.to(DEV)
    # eval(): dropout off, the same as p = 0
    stack, dense = _model(D, dtype, 111)
    stack.eval()
    r1 = _run(stack, dense, xd, graph, anchor, dist, targets, pairs)
    stack.dropout_p = 0.0
    r2 = _run(stack, dense, xd, graph, anchor, dist, targets, pairs)
    _bitwise_equal(r1, r2)
    # ungated: the block ignores dropout, as on the unpaired path
    stack, dense = _model(D, dtype, 112, gated=False)
    r1 = _run(stack, dense, xd, graph, anchor, dist, targets, pairs)
    stack.dropout_p = 0.0
    r2 = _run(stack, dense, xd, graph, anchor, dist, targets, pairs)
    _bitwise_equal(r1, r2)
    # without the opt-in, train-mode dropout on pairs is still refused
    stack, dense = _model(D, dtype, 113, pair_dropout=False)
    with pytest.raises(E.EdgError, match="gate dropout"):
        _run(stack, dense, xd, graph, anchor, dist, targets, pairs)
    # no pairs at all: runs, and the gates get zero gradients
    stack, dense = _model(D, dtype, 114)
    none = E.pairs_from_ptr(graph, torch.zeros(batch.n_graphs + 1, dtype=torch.int32),
                            torch.zeros(0, dtype=torch.int32))
    a0 = torch.zeros(0, dtype=torch.int32, device=DEV)
    d0 = E.tree_distance(graph, a0, pairs=none)
    xg = xd.clone().requires_grad_(True)
    out = stack(xg, graph, a0, d0, lambda a, q: dense(torch.cat([a, q], 1)), head_params=list(dense.parameters()),
                pairs=none)
    assert out.logits.shape == (0, 34)
    (out.logits.sum() + out.xy + out.kl).backward()
    for n, p in stack.named_parameters():
        if n.startswith("gate"):
            assert p.grad is not None and float(p.grad.abs().max()) == 0.0, n


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
def test_two_runs_with_the_same_seed_are_bitwise_equal(dtype):
    batch, pp, an = _layout("windows")
    D = 64
    stack, dense = _model(D, dtype, 121)
    graph, pairs, anchor, dist, x, targets = _inputs(batch, pp, an, D, 121)
    runs = []
    for _ in range(2):
        torch.manual_seed(5)
        runs.append(_run(stack, dense, x.to(DEV), graph, anchor, dist, targets, pairs))
    _bitwise_equal(*runs)
    torch.manual_seed(6)
    r3 = _run(stack, dense, x.to(DEV), graph, anchor, dist, targets, pairs)
    assert not torch.equal(r3[0].view_arg, runs[0][0].view_arg)        # another seed, other masks


def test_captured_dropout_step_replays_the_seed_it_reads(monkeypatch):
    """Graph build, pairs_from_ptr(n_pair_rows=), tree_distance(pairs=) and the dropout training step with a DenseHead
    and total_loss in one CUDA graph (a device->host read during capture raises).  The seed comes from a static device
    tensor: each replay equals the eager run with the seed written into it."""
    import ed_gated_gcn_b200 as E
    from ed_gated_gcn_b200 import gated, synth
    from ed_gated_gcn_b200.runtime import GraphedStep
    batch = synth.config_batch("C2", n_graphs=96)
    pp, an = synth.candidate_pairs(batch)
    D = 300
    stack, _ = _model(D, torch.bfloat16, 131)
    head = E.DenseHead(2 * D, 34).to(DEV)
    seed_t = torch.zeros(1, dtype=torch.int64, device=DEV)
    monkeypatch.setattr(gated, "_dropout_seed", lambda device: seed_t)
    st = dict(h=torch.from_numpy(batch.heads).to(DEV), sp=torch.from_numpy(batch.sent_ptr).to(DEV),
              pp=torch.from_numpy(pp).to(DEV), an=torch.from_numpy(an).to(DEV),
              tg=(torch.arange(len(an)) % 34).to(DEV))
    x = torch.randn(batch.n_rows, D, generator=torch.Generator().manual_seed(132)).to(DEV).requires_grad_(True)
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
        res.update(loss=loss.detach(), logits=out.logits.detach(), scores=out.scores.detach(),
                   view_arg=out.view_arg.detach(), dx=x.grad, gw=stack.gc1.weight.grad,
                   gate_w=stack.gate1[1].weight.grad)
        return loss

    seeds = (0x1234_5678_9ABC_DEF, 0x0FED_CBA9_8765_432)
    eager = []
    for s in seeds:
        seed_t.fill_(s)
        step()
        eager.append({k: v.clone() for k, v in res.items()})
    gs = GraphedStep(step)
    for s, want in zip(seeds, eager):
        seed_t.fill_(s)
        gs()
        torch.cuda.synchronize()
        for k, v in want.items():
            assert torch.equal(res[k], v), (hex(s), k)
    assert not torch.equal(eager[0]["view_arg"], eager[1]["view_arg"])
    assert not torch.equal(eager[0]["dx"], eager[1]["dx"])
