"""BertAmir54's sigmoid fc head on grouped trigger pairs (``GatedGCNStack(fc_sigmoid=True, pair_fc_sigmoid=True)``,
``pairs=``).

Each pair's scores read ``z = sigmoid(g_p * h_t)`` (bert_amir5.py:464-465, :538), formed per (pair, row) from the
sentence rows.  References: the reference's own BertAmir54 run (golden block54) through the pairs path with one pair per
sentence, the existing stack on the expanded batch (each sentence copied once per pair), and the oracle run once per
pair (``gated_block_ref(fc_sigmoid=True)``, in fp64), with the dropout masks rebuilt in numpy where gate dropout is on.

``fc.1.weight`` is judged as in the golden BertAmir54 test: its gradient sums ``ds_t * sigmoid(...)`` with
``sum_t ds_t = 0``, a cancelling sum, so besides the relative tolerance it may miss by the error bound of that sum (a
few dozen roundings of the compute dtype on ``sum |summand|``).  ``fc.1.bias`` cancels inside the softmax and is skipped,
as ``fc.0.bias`` is everywhere else."""
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN
from gpu_util import DEV, rel, tol_for
from oracle import fixtures, ref_oracle as O
from test_gpu_c_models import _check_routing, _compare, _dropout_mask_numpy, _fp64_fc_weight_grad_block54
from test_gpu_j_pairs import _dense_of, _expand, _expand_dist, _graph, _layout, _oracle_dx_per_sentence, _sum_dx
from test_gpu_k_pairs_dropout import _bitwise_equal, _check_args_equal

pytestmark = pytest.mark.gpu

P_DROP = 0.25
EPS = {torch.float32: 2.0 ** -23, torch.bfloat16: 2.0 ** -8}
ROUNDINGS = {torch.float32: 64, torch.bfloat16: 8}


def _model(D, dtype, seed, Lyr=2, p=0.0, C=34, **kw):
    import ed_gated_gcn_b200 as E
    torch.manual_seed(seed)
    kw.setdefault("pair_fc_sigmoid", True)
    stack = E.GatedGCNStack(D, n_layers=Lyr, n_classes=C, compute_dtype=dtype, fc_sigmoid=True, dropout=p,
                            pair_dropout=p > 0, **kw).to(DEV)
    stack.train(p > 0)
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


def _run(stack, head, x0, graph, anchor, dist, targets, pairs=None, score_w=None):
    """One training step; ``head`` is an nn.Linear (torch lambda head) or a DenseHead.  ``score_w``: the loss also
    takes ``sum(scores * score_w)`` (the scores then carry their own gradient)."""
    import ed_gated_gcn_b200 as E
    for p in list(stack.parameters()) + list(head.parameters()):
        p.grad = None
    x = x0.clone().requires_grad_(True)
    if isinstance(head, E.DenseHead):
        out = stack(x, graph, anchor, dist, head, pairs=pairs)
        loss = E.cross_entropy(out.logits, targets.to(DEV)) + 0.01 * out.xy + 0.01 * out.kl
    else:
        out = stack(x, graph, anchor, dist, lambda a, q: head(torch.cat([a, q], 1)), head_params=list(head.parameters()),
                    pairs=pairs)
        loss = torch.nn.functional.cross_entropy(out.logits, targets.to(DEV)) + 0.01 * out.xy + 0.01 * out.kl
    if score_w is not None:
        loss = loss + (out.scores * score_w).sum()
    loss.backward()
    grads = {n: p.grad.detach().clone() for n, p in list(stack.named_parameters()) + [("dense.weight", head.weight),
                                                                                   ("dense.bias", head.bias)]
             if p.grad is not None}
    return out, loss.detach(), x.grad.detach(), grads


def _fc_scale(out, pairs, dist, kl_w=0.01):
    """An upper bound (sigmoid <= 1) of max_cj sum_pt |ds_pt logits_pc sigmoid(cat)_ptj| from a run whose loss takes
    ``kl_w * kl``, with ds_pt = kl_w / P * P_pt (Q_pt - kl_p) rebuilt from its scores and distances: the scale of
    fc.1.weight's cancelling sum where no oracle runs."""
    P = pairs.n_pairs
    lens = (pairs.pair_row_ptr[1:] - pairs.pair_row_ptr[:-1]).long()
    owner = torch.repeat_interleave(torch.arange(P, device=lens.device), lens)
    zeros = torch.zeros(P, dtype=torch.float64, device=lens.device)

    def softmax(v):
        m = torch.full_like(zeros, -float("inf")).scatter_reduce(0, owner, v, "amax")
        e = (v - m[owner]).exp()
        return e / zeros.index_add(0, owner, e)[owner]

    ps, qs = softmax(out.scores.detach().double()), softmax(dist.double())
    ds = kl_w / P * ps * (qs - zeros.index_add(0, owner, ps * qs)[owner])
    per_pair = zeros.index_add(0, owner, ds.abs())
    return float((out.logits.detach().double().abs() * per_pair[:, None]).sum(0).max())


def _fc_weight_ok(got, want, sum_abs, tol, dtype):
    err = (got.detach().double().cpu() - want.detach().double().cpu()).abs().max().item()
    bound = max(tol * want.detach().double().abs().max().item(), ROUNDINGS[dtype] * EPS[dtype] * sum_abs)
    return err <= bound, (err, bound)


def _oracle54(stack, dense, batch, pp, an, x, dist, targets, forced=None, masks=None):
    """``gated_block_ref(fc_sigmoid=True)`` once per pair in fp64; ``forced`` = (final_arg [P,D], view_arg [V,P,D]) as
    sentence-local rows, ``masks`` = per stream [n_pair_rows, D] dropout masks.  Also returns max_cj of
    sum_pt |ds_pt logits_pc sigmoid(cat)_ptj| (the scale of fc.1.weight's cancelling sum)."""
    dt = torch.float64
    sd = {k: v.detach().cpu().to(dt).requires_grad_(True) for k, v in stack.state_dict().items()}
    dw = dense.weight.detach().cpu().to(dt).requires_grad_(True)
    db = dense.bias.detach().cpu().to(dt).requires_grad_(True)
    lead, n_lin = O.GATE_ARCHS[stack.gate_arch]
    off = 1 if lead else 0
    Lyr = stack.n_layers
    gcn_p = [(sd[f"gc{l}.weight"], sd[f"gc{l}.bias"]) for l in range(1, Lyr + 1)]
    gate_p = [[(sd[f"gate{l}.{off + 2 * i}.weight"], sd[f"gate{l}.{off + 2 * i}.bias"]) for i in range(n_lin)]
              for l in range(1, Lyr + 1)]
    sp = batch.sent_ptr
    owner = np.repeat(np.arange(batch.n_graphs), np.diff(pp))
    dc = dist.cpu().long()
    P = len(an)
    xs, logits, scores, outs = [], [], [], []
    views_vals, final_vals = [], []
    xy = kl = 0.0
    o = 0
    for p, s in enumerate(owner):
        lo, hi = int(sp[s]), int(sp[s + 1])
        n = hi - lo
        xb = x[lo:hi].to(dt).clone().requires_grad_(True)
        adj = torch.from_numpy(_dense_of(batch, s)).to(dt)
        r = O.gated_block_ref(xb[None], adj[None], torch.tensor([int(an[p])]), dc[o:o + n][None], gcn_p, gate_p,
                              sd["fc.1.weight"], sd["fc.1.bias"], lambda a, q: torch.cat([a, q], 1) @ dw.t() + db,
                              lead_sigmoid=lead, fc_sigmoid=True,
                              forced_view_arg=None if forced is None else forced[1][:, p:p + 1],
                              forced_final_arg=None if forced is None else forced[0][p:p + 1],
                              gate_masks=None if masks is None else [m[o:o + n][None].to(dt) for m in masks])
        r["scores"].retain_grad()
        xs.append(xb); logits.append(r["logits"]); scores.append(r["scores"][0]); outs.append(r)
        views_vals.append([(r["hs"][0][0] * g[0][None, :]).detach() for g in r["gates"]])
        final_vals.append(r["x_out"][0].detach())
        xy = xy + r["xy"] / P
        kl = kl + r["kl"] / P
        o += n
    lg = torch.cat(logits)
    loss = torch.nn.functional.cross_entropy(lg, targets) + 0.01 * xy + 0.01 * kl
    loss.backward()
    D = x.shape[1]
    sum_abs = torch.zeros(stack.n_classes, 2 * D, dtype=dt)
    for r in outs:
        n = r["x_out"].shape[1]
        cat = torch.sigmoid(torch.cat([r["x_out"].detach(), r["aspect"].detach()[:, None, :].expand(1, n, D)], 2))[0]
        sum_abs += torch.einsum("t,c,tj->cj", r["scores"].grad[0].abs(), r["logits"].detach()[0].abs(), cat)
    grads = {k: v.grad for k, v in sd.items()}
    grads["dense.weight"], grads["dense.bias"] = dw.grad, db.grad
    ora = dict(logits=lg, scores=scores, xy=xy, kl=kl, loss=loss, dx=[t.grad for t in xs], grads=grads,
               views_vals=views_vals, final_vals=final_vals, fc_sum_abs=sum_abs.max().item())
    return ora, owner


def _compare_oracle(res, stack, dense, batch, ora, owner, ora_g, tol, dtype):
    """_compare with fc.1.weight judged by :func:`_fc_weight_ok` and fc.1.bias skipped."""
    out, loss, dx, _ = res
    og = _oracle_dx_per_sentence(ora_g, owner, batch)
    fc_w = og["grads"]["fc.1.weight"]
    og["grads"] = dict(og["grads"], **{"fc.1.weight": None, "fc.1.bias": None})
    _compare(out, loss, dx, stack, dense, ora, og, tol, stack.n_layers)
    ok, why = _fc_weight_ok(stack.fc[1].weight.grad, fc_w, ora_g["fc_sum_abs"], tol, dtype)
    assert ok, why


def _compare_expanded(res_g, res_e, rows, N, tol, fc_sum_abs, dtype):
    out, loss, dx, grads = res_g
    oe, le, dxe, ge = res_e
    for k in ("logits", "pooled", "scores"):
        assert rel(getattr(out, k), getattr(oe, k)) < tol, k
    assert rel(out.xy, oe.xy) < tol and rel(out.kl, oe.kl) < tol and rel(loss, le) < tol
    assert rel(dx.double().cpu(), _sum_dx(dxe, rows, N)) < tol, "dx"
    for n, g in ge.items():
        if n == "fc.1.bias" or g.abs().max() < 1e-9:
            continue
        if n == "fc.1.weight":                 # both sides carry the cancelling sum's error: twice the bound
            ok, why = _fc_weight_ok(grads[n], g, 2 * fc_sum_abs, tol, dtype)
            assert ok, why
            continue
        assert rel(grads[n], g) < tol, n


def _expanded_run(stack, dense, batch, pp, an, x, targets, **kw):
    eb, rows = _expand(batch, pp, an)
    eg = _graph(eb)
    ea = torch.from_numpy(eb.anchor).to(DEV)
    return _run(stack, dense, x[rows].to(DEV), eg, ea, _expand_dist(eg, ea), targets, **kw), rows


# ------------------------------------------------------------------------------------------------ tests
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
def test_block54_golden_through_pairs(dtype):
    """The reference's own BertAmir54.forward + backward (golden block54) through pairs= with one pair per sentence:
    the dense-compat batch as sentence rows, every sentence's trigger its one pair."""
    import ed_gated_gcn_b200 as E
    z = fixtures.load(os.path.join(GOLDEN, "block54.npz"))
    tol = tol_for(dtype)
    C, D2 = z["p_fc.1.weight"].shape
    D = D2 // 2
    stack = E.GatedGCNStack(D, n_layers=2, n_classes=C, gate_arch="sig-2", compute_dtype=dtype, fc_sigmoid=True,
                            pair_fc_sigmoid=True).to(DEV)
    stack.load_state_dict({k[2:]: torch.from_numpy(z[k]) for k in z if k.startswith("p_") and not k.startswith("p_dense.")})
    dense = torch.nn.Sequential(torch.nn.Linear(2 * D + 768, 768), torch.nn.Linear(768, C)).to(DEV)
    dense.load_state_dict({k[len("p_dense."):]: torch.from_numpy(z[k]) for k in z if k.startswith("p_dense.")})
    B, T, _ = z["x"].shape
    x = torch.from_numpy(z["x"]).reshape(B * T, D).to(DEV).requires_grad_(True)
    graph = E.graph_from_dense(torch.from_numpy(z["adj"]).to(DEV))
    anchor = torch.from_numpy(z["anchor"]).to(DEV)
    pairs = E.pairs_from_ptr(graph, torch.arange(B + 1, dtype=torch.int32), torch.from_numpy(z["anchor"]).int())
    dist = torch.from_numpy(z["dist"]).reshape(-1).to(DEV)          # one pair per sentence: per-pair packed = the rows
    pooled_output = torch.from_numpy(z["dense_in"][:, 2 * D:]).to(DEV)
    out = stack(x, graph, anchor, dist, lambda a, p: dense(torch.cat([a, p, pooled_output], dim=1)),
                head_params=list(dense.parameters()), pairs=pairs)
    loss = torch.nn.functional.cross_entropy(out.logits, torch.from_numpy(z["targets"]).to(DEV)) + 0.01 * out.xy \
        + 0.01 * out.kl
    loss.backward()
    assert rel(out.logits, z["logits"]) < tol
    assert rel(out.scores.reshape(B, T), z["scores"]) < tol
    assert rel(out.xy, z["xy"]) < tol and rel(out.kl, z["kl"]) < tol and rel(loss, z["loss"]) < tol
    if dtype != torch.float32:
        return                                     # bf16 gradients: the routing rule of DESIGN 4 (oracle tests below)
    assert rel(x.grad.reshape(B, T, D), z["dx"]) < tol
    got = dict(stack.named_parameters())
    got.update({"dense." + n: p for n, p in dense.named_parameters()})
    for k in z:
        if k.startswith("g_") and k not in ("g_fc.1.bias", "g_fc.1.weight"):
            assert rel(fixtures.pick(z, k, got[k[2:]].grad), z[k]) < tol, k
    g64, sum_abs = _fp64_fc_weight_grad_block54(z)
    err = (got["fc.1.weight"].grad.detach().cpu().double() - g64).abs().max().item()
    assert err < 64 * 1.1920929e-07 * sum_abs, err


@pytest.mark.parametrize("layout", ["mixed", "windows", "long", "extra"])
def test_fp32_vs_oracle_and_expanded(layout):
    batch, pp, an = _layout(layout)
    D = 64
    stack, dense = _model(D, torch.float32, 11)
    graph, pairs, anchor, dist, x, targets = _inputs(batch, pp, an, D, 11)
    res = _run(stack, dense, x.to(DEV), graph, anchor, dist, targets, pairs)
    ora, owner = _oracle54(stack, dense, batch, pp, an, x, dist, targets)
    _compare_oracle(res, stack, dense, batch, ora, owner, ora, 1e-5, torch.float32)
    res_e, rows = _expanded_run(stack, dense, batch, pp, an, x, targets)
    _compare_expanded(res, res_e, rows, batch.n_rows, 1e-4, ora["fc_sum_abs"], torch.float32)
    assert ora["fc_sum_abs"] <= _fc_scale(res[0], pairs, dist) * (1 + 1e-4)


@pytest.mark.parametrize("fused", [True, False], ids=["fused", "unfused"])
@pytest.mark.parametrize("layout", ["mixed", "windows", "extra"])
def test_bf16_vs_oracle(layout, fused, monkeypatch):
    """bf16 on the fused chain (which the sigmoid head no longer rules out on pairs) and on the unfused kernels, against
    the oracle under this path's max-pool routing."""
    from ed_gated_gcn_b200 import gated
    from test_gpu_g_fused_limits import _spy_fused_plan
    monkeypatch.setattr(gated, "_FUSED", fused)
    seen = _spy_fused_plan(monkeypatch)
    batch, pp, an = _layout(layout)
    D = 64
    stack, dense = _model(D, torch.bfloat16, 21)
    graph, pairs, anchor, dist, x, targets = _inputs(batch, pp, an, D, 21)
    res = _run(stack, dense, x.to(DEV), graph, anchor, dist, targets, pairs)
    assert (seen[0] is not None) == fused
    ora, owner = _oracle54(stack, dense, batch, pp, an, x, dist, targets)
    starts = torch.from_numpy(batch.sent_ptr[:-1][owner].astype(np.int64))
    ora_g, _ = _oracle54(stack, dense, batch, pp, an, x, dist, targets, forced=_check_routing(res[0], ora, starts))
    _compare_oracle(res, stack, dense, batch, ora, owner, ora_g, 2e-2, torch.bfloat16)


@pytest.mark.parametrize("Lyr", [2, 3])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
@pytest.mark.parametrize("layout", ["mixed", "extra"])
def test_dropout_vs_expanded_same_seed(layout, dtype, Lyr, monkeypatch):
    if dtype == torch.float32:
        monkeypatch.setenv("EDG_F32_TC", "0")       # one projection kernel in both arms (test_gpu_k_pairs_dropout)
    batch, pp, an = _layout(layout)
    D = 64
    seed = 71 + Lyr
    stack, dense = _model(D, dtype, seed, Lyr=Lyr, p=P_DROP)
    graph, pairs, anchor, dist, x, targets = _inputs(batch, pp, an, D, seed)
    torch.manual_seed(seed + 3)
    res_g = _run(stack, dense, x.to(DEV), graph, anchor, dist, targets, pairs)
    seed_g = int(stack.last_dropout_seed)
    torch.manual_seed(seed + 3)
    res_e, rows = _expanded_run(stack, dense, batch, pp, an, x, targets)
    assert seed_g == int(stack.last_dropout_seed)
    _check_args_equal(res_g[0], res_e[0], rows)
    _compare_expanded(res_g, res_e, rows, batch.n_rows, 1e-4 if dtype == torch.float32 else 2e-2,
                      _fc_scale(res_g[0], pairs, dist), dtype)


@pytest.mark.parametrize("Lyr", [2, 3])
@pytest.mark.parametrize("layout", ["mixed", "extra"])
def test_dropout_vs_oracle_f32(layout, Lyr):
    batch, pp, an = _layout(layout)
    D = 64
    stack, dense = _model(D, torch.float32, 81, Lyr=Lyr, p=P_DROP)
    graph, pairs, anchor, dist, x, targets = _inputs(batch, pp, an, D, 81)
    res = _run(stack, dense, x.to(DEV), graph, anchor, dist, targets, pairs)
    masks = [torch.from_numpy(_dropout_mask_numpy(int(stack.last_dropout_seed), v, P_DROP, pairs.n_pair_rows, D))
             for v in range(Lyr)]
    ora, owner = _oracle54(stack, dense, batch, pp, an, x, dist, targets, masks=masks)
    _compare_oracle(res, stack, dense, batch, ora, owner, ora, 1e-5, torch.float32)


@pytest.mark.parametrize("drop", [False, True], ids=["eval", "dropout"])
def test_dense_head_matches_torch_head(drop):
    """The block's own head kernels (DenseHead + E.cross_entropy) against the same head as a torch lambda."""
    import ed_gated_gcn_b200 as E
    batch, pp, an = _layout("mixed")
    D = 64
    stack, dense = _model(D, torch.float32, 141, p=P_DROP if drop else 0.0)
    head = E.DenseHead(2 * D, 34).to(DEV)
    with torch.no_grad():
        head.weight.copy_(dense.weight)
        head.bias.copy_(dense.bias)
    graph, pairs, anchor, dist, x, targets = _inputs(batch, pp, an, D, 141)
    torch.manual_seed(5)
    r_t = _run(stack, dense, x.to(DEV), graph, anchor, dist, targets, pairs)
    torch.manual_seed(5)
    r_d = _run(stack, head, x.to(DEV), graph, anchor, dist, targets, pairs)
    for k in ("logits", "scores", "pooled", "xy", "kl"):
        assert rel(getattr(r_d[0], k), getattr(r_t[0], k)) < 1e-5, k
    assert rel(r_d[1], r_t[1]) < 1e-5 and rel(r_d[2], r_t[2]) < 1e-5
    for n, g in r_t[3].items():
        if n != "fc.1.bias":
            assert rel(r_d[3][n], g) < 1e-5, n


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
@pytest.mark.parametrize("drop", [False, True], ids=["eval", "dropout"])
def test_scores_carrying_gradient_vs_expanded(drop, dtype, monkeypatch):
    """A loss that also reads out.scores: the head backward takes g_scores (its first pass gives d v, d c).  Both arms
    run the same projection kernels (EDG_F32_TC=0 in fp32, the unfused chain in bf16, which unpaired BertAmir54 always
    uses), so they compute the same rows and route the max-pools alike."""
    from ed_gated_gcn_b200 import gated
    if dtype == torch.float32:
        monkeypatch.setenv("EDG_F32_TC", "0")
    else:
        monkeypatch.setattr(gated, "_FUSED", False)
    batch, pp, an = _layout("windows")
    D = 64
    stack, dense = _model(D, dtype, 151, p=P_DROP if drop else 0.0)
    graph, pairs, anchor, dist, x, targets = _inputs(batch, pp, an, D, 151)
    w = torch.randn(pairs.n_pair_rows, generator=torch.Generator().manual_seed(152)).to(DEV) * 0.05
    torch.manual_seed(7)
    res_g = _run(stack, dense, x.to(DEV), graph, anchor, dist, targets, pairs, score_w=w)
    torch.manual_seed(7)
    res_e, rows = _expanded_run(stack, dense, batch, pp, an, x, targets, score_w=w)   # same per-pair packed row order
    tol = 1e-4 if dtype == torch.float32 else 2e-2
    out, loss, dx, grads = res_g
    assert rel(out.scores, res_e[0].scores) < tol and rel(loss, res_e[1]) < tol
    assert rel(dx.double().cpu(), _sum_dx(res_e[2], rows, batch.n_rows)) < tol, "dx"
    for n, g in res_e[3].items():
        if n not in ("fc.1.bias", "fc.1.weight") and g.abs().max() > 1e-9:
            assert rel(grads[n], g) < tol, n
    # the scores' own gradient does not cancel: fc.1.weight is held to the plain tolerance here
    assert rel(grads["fc.1.weight"], res_e[3]["fc.1.weight"]) < tol


def test_512_token_sentence_with_512_pairs_vs_expanded():
    batch, pp, an = _layout("512")
    D = 64
    stack, dense = _model(D, torch.float32, 41)
    graph, pairs, anchor, dist, x, targets = _inputs(batch, pp, an, D, 41)
    res = _run(stack, dense, x.to(DEV), graph, anchor, dist, targets, pairs)
    res_e, rows = _expanded_run(stack, dense, batch, pp, an, x, targets)
    _compare_expanded(res, res_e, rows, batch.n_rows, 1e-4, _fc_scale(res[0], pairs, dist), torch.float32)


@pytest.mark.parametrize("drop", [False, True], ids=["eval", "dropout"])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
def test_no_pairs(dtype, drop):
    """A batch without pairs (P = 0): runs, the logits are empty, dx and the gate gradients are zero.  Sentences
    without pairs next to ones with pairs are part of the "mixed" layout above."""
    import ed_gated_gcn_b200 as E
    batch, pp, an = _layout("mixed")
    D = 64
    stack, dense = _model(D, dtype, 161, p=P_DROP if drop else 0.0)
    graph = _graph(batch)
    none = E.pairs_from_ptr(graph, torch.zeros(batch.n_graphs + 1, dtype=torch.int32), torch.zeros(0, dtype=torch.int32))
    a0 = torch.zeros(0, dtype=torch.int32, device=DEV)
    d0 = E.tree_distance(graph, a0, pairs=none)
    x = torch.randn(batch.n_rows, D, device=DEV).requires_grad_(True)
    out = stack(x, graph, a0, d0, lambda a, q: dense(torch.cat([a, q], 1)), head_params=list(dense.parameters()),
                pairs=none)
    assert out.logits.shape == (0, 34) and out.scores.shape == (0,)
    (out.logits.sum() + out.xy + out.kl).backward()
    assert float(x.grad.abs().max()) == 0.0
    for n, p in stack.named_parameters():
        if n.startswith("gate"):
            assert p.grad is not None and float(p.grad.abs().max()) == 0.0, n


@pytest.mark.parametrize("drop", [False, True], ids=["eval", "dropout"])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
def test_two_runs_are_bitwise_equal(dtype, drop):
    batch, pp, an = _layout("windows")
    D = 64
    stack, dense = _model(D, dtype, 171, p=P_DROP if drop else 0.0)
    graph, pairs, anchor, dist, x, targets = _inputs(batch, pp, an, D, 171)
    runs = []
    for _ in range(2):
        torch.manual_seed(5)
        runs.append(_run(stack, dense, x.to(DEV), graph, anchor, dist, targets, pairs))
    _bitwise_equal(*runs)


def test_captured_dropout_step_replays_the_seed_it_reads(monkeypatch):
    """Graph build, pairs_from_ptr(n_pair_rows=), tree_distance(pairs=) and the BertAmir54 dropout training step with a
    DenseHead in one CUDA graph; the seed comes from a static device tensor and each replay equals the eager run."""
    import ed_gated_gcn_b200 as E
    from ed_gated_gcn_b200 import gated, synth
    from ed_gated_gcn_b200.runtime import GraphedStep
    batch = synth.config_batch("C2", n_graphs=96)
    pp, an = synth.candidate_pairs(batch)
    D = 256
    stack, _ = _model(D, torch.bfloat16, 181, p=P_DROP)
    head = E.DenseHead(2 * D, 34).to(DEV)
    seed_t = torch.zeros(1, dtype=torch.int64, device=DEV)
    monkeypatch.setattr(gated, "_dropout_seed", lambda device: seed_t)
    st = dict(h=torch.from_numpy(batch.heads).to(DEV), sp=torch.from_numpy(batch.sent_ptr).to(DEV),
              pp=torch.from_numpy(pp).to(DEV), an=torch.from_numpy(an).to(DEV),
              tg=(torch.arange(len(an)) % 34).to(DEV))
    x = torch.randn(batch.n_rows, D, generator=torch.Generator().manual_seed(182)).to(DEV).requires_grad_(True)
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
                   gw=stack.gc1.weight.grad, fc_w=stack.fc[1].weight.grad, gate_w=stack.gate2[1].weight.grad)
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
    assert not torch.equal(eager[0]["scores"], eager[1]["scores"])


def test_switch_scope_and_declined_combinations():
    """Without pair_fc_sigmoid the refusal stays and names the switch; the switch changes nothing without fc_sigmoid
    or without pairs=; view_len, aspect and return_x_out stay declined with it on."""
    import ed_gated_gcn_b200 as E
    from ed_gated_gcn_b200 import synth
    batch, pp, an = _layout("mixed")
    D = 64
    graph, pairs, anchor, dist, x, targets = _inputs(batch, pp, an, D, 191)
    xd = x.to(DEV)
    stack, dense = _model(D, torch.bfloat16, 191, pair_fc_sigmoid=False)
    with pytest.raises(E.EdgError, match="pair_fc_sigmoid"):
        _run(stack, dense, xd, graph, anchor, dist, targets, pairs)
    # no effect on the unpaired path
    ub = synth.make_batch(8, 3, 20, seed=192)
    ug = _graph(ub)
    ua = torch.from_numpy(ub.anchor).to(DEV)
    ux = torch.randn(ub.n_rows, D, generator=torch.Generator().manual_seed(193)).to(DEV)
    ut = torch.arange(ub.n_graphs) % 34
    r1 = _run(stack, dense, ux, ug, ua, E.tree_distance(ug, ua), ut)
    stack.pair_fc_sigmoid = True
    _bitwise_equal(r1, _run(stack, dense, ux, ug, ua, E.tree_distance(ug, ua), ut))
    # no effect without fc_sigmoid
    torch.manual_seed(192)
    plain = E.GatedGCNStack(D, n_classes=34, compute_dtype=torch.bfloat16).to(DEV)
    torch.manual_seed(192)
    switched = E.GatedGCNStack(D, n_classes=34, compute_dtype=torch.bfloat16, pair_fc_sigmoid=True).to(DEV)
    _bitwise_equal(_run(plain, dense, xd, graph, anchor, dist, targets, pairs),
                   _run(switched, dense, xd, graph, anchor, dist, targets, pairs))
    fn = lambda a, q: dense(torch.cat([a, q], 1))
    for kw, match in ((dict(view_len=torch.ones(batch.n_graphs, dtype=torch.int64, device=DEV)), "view_len"),
                      (dict(aspect=torch.zeros(len(an), D, device=DEV)), "aspect"),
                      (dict(return_x_out=True), "return_x_out")):
        with pytest.raises(E.EdgError, match=match):
            stack(xd, graph, anchor, dist, fn, head_params=list(dense.parameters()), pairs=pairs, **kw)
