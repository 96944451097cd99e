"""Module-level parity: the drop-in GraphConvolution and the fused GatedGCNStack against
(a) the fixtures the reference itself produced (tests/golden) and (b) the CPU oracle on
seeded synthetic batches.  fp32: <= 1e-5 relative; bf16: <= 2e-2 relative (north_star)."""
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN
from gpu_util import DEV, rel, tol_for, dense_inputs, pack_rows
from oracle import fixtures, ref_oracle as O

pytestmark = pytest.mark.gpu
DTYPES = [torch.float32, torch.bfloat16]


# ------------------------------------------------------------------------- GraphConvolution
@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "bf16"])
def test_graph_convolution_matches_reference_outputs(dtype):
    """models/gcn.py run by the reference itself (golden) vs the drop-in module, dense interface."""
    import ed_gated_gcn_b200 as E
    z = fixtures.load(os.path.join(GOLDEN, "gcn_layer.npz"))
    tol = tol_for(dtype)
    for ci in range(int(z["n_cases"])):
        p = f"c{ci}_"
        T = int(z[p + "T"])
        sp = z[p + "sent_ptr"]
        heads = [z[p + "heads"][sp[b]:sp[b + 1]] for b in range(len(sp) - 1)]
        full = torch.from_numpy(np.stack([O.dense_adjacency_from_heads(h, 100) for h in heads])).float().to(DEV)
        adj = full[:, :T, :T]                                        # bert_amir5.py:589
        has_bias = (p + "bias") in z
        Din, Dout = z[p + "weight"].shape
        layer = E.GraphConvolution(Din, Dout, None, bias=has_bias, compute_dtype=dtype).to(DEV)
        with torch.no_grad():
            layer.weight.copy_(torch.from_numpy(z[p + "weight"]))
            if has_bias:
                layer.bias.copy_(torch.from_numpy(z[p + "bias"]))
        text = torch.from_numpy(z[p + "text"]).to(DEV).requires_grad_(True)
        y = layer(text, adj)
        assert y.shape == (len(heads), T, Dout) and y.dtype == torch.float32
        (y * torch.from_numpy(z[p + "probe"]).to(DEV)).sum().backward()
        assert rel(y, z[p + "y"]) < tol, ci
        assert rel(text.grad, z[p + "dtext"]) < tol, ci
        assert rel(layer.weight.grad, z[p + "dweight"]) < tol, ci
        if has_bias:
            assert rel(layer.bias.grad, z[p + "dbias"]) < tol, ci


def test_graph_convolution_two_layers_share_one_csr_and_state_dict_keys():
    import ed_gated_gcn_b200 as E
    from ed_gated_gcn_b200 import gcn as G
    from ed_gated_gcn_b200 import synth
    batch = synth.make_batch(5, 3, 12, seed=2)
    x, adj, T = dense_inputs(batch, 24, seed=2)
    m = torch.nn.Module()
    m.gc1 = E.GraphConvolution(24, 24, None)
    m.gc2 = E.GraphConvolution(24, 24, None)
    m.to(DEV)
    assert set(m.state_dict()) == {"gc1.weight", "gc1.bias", "gc2.weight", "gc2.bias"}
    assert m.gc1.weight.shape == (24, 24)                             # [in,out], gcn.py:18
    adj_d = adj.to(DEV)
    G._GRAPH_CACHE.clear()
    h1 = m.gc1(x.to(DEV), adj_d)
    h2 = m.gc2(h1, adj_d)
    assert len(G._GRAPH_CACHE) == 1
    w1, b1, w2, b2 = (t.detach().cpu() for t in (m.gc1.weight, m.gc1.bias, m.gc2.weight, m.gc2.bias))
    want = O.gcn_layer_ref(O.gcn_layer_ref(x, adj, w1, b1), adj, w2, b2)
    assert rel(h2, want) < 1e-5


def test_graph_convolution_cache_never_returns_a_stale_graph():
    """train.py:108 makes a fresh `.to(device)` adjacency per batch: the caching allocator hands the freed block to the
    next batch at the same address, same shape, version 0.  The CSR cache must key on the tensor OBJECT, not its address."""
    import ed_gated_gcn_b200 as E
    from ed_gated_gcn_b200 import gcn as G
    from ed_gated_gcn_b200 import synth
    layer = E.GraphConvolution(16, 16, None).to(DEV)
    w, b = layer.weight.detach().cpu(), layer.bias.detach().cpu()
    seen_ptrs = set()
    for seed in (21, 22, 23, 24):
        batch = synth.make_batch(6, 12, 12, seed=seed)                # same shapes every time, different trees
        x, adj, T = dense_inputs(batch, 16, seed=seed)
        adj_d = adj.to(DEV)
        seen_ptrs.add(adj_d.data_ptr())
        y = layer(x.to(DEV), adj_d)
        assert rel(y, O.gcn_layer_ref(x, adj, w, b)) < 1e-5, seed
        # an in-place edit of the same object must miss as well
        adj_d[:, 0, 1] = 1.0; adj_d[:, 1, 0] = 1.0
        adj2 = adj.clone(); adj2[:, 0, 1] = 1.0; adj2[:, 1, 0] = 1.0
        assert rel(layer(x.to(DEV), adj_d), O.gcn_layer_ref(x, adj2, w, b)) < 1e-5, seed
        del adj_d, y
    assert len(G._GRAPH_CACHE) == 0                                  # entries die with their tensors
    assert len(seen_ptrs) < 4                                        # the allocator did reuse an address (the bug's precondition)


def test_graph_convolution_relu_option_defaults_off():
    import ed_gated_gcn_b200 as E
    from ed_gated_gcn_b200 import synth
    batch = synth.make_batch(4, 3, 9, seed=9)
    x, adj, T = dense_inputs(batch, 16, seed=9)
    layer = E.GraphConvolution(16, 16, None).to(DEV)
    assert layer.relu is False
    y = layer(x.to(DEV), adj.to(DEV))
    assert (y < 0).any()                                              # no non-linearity (gcn.py:19 is dead code)
    layer_r = E.GraphConvolution(16, 16, None, relu=True).to(DEV)
    layer_r.load_state_dict(layer.state_dict())
    xr = x.to(DEV).requires_grad_(True)
    yr = layer_r(xr, adj.to(DEV))
    assert torch.equal(yr, torch.relu(y))
    yr.sum().backward()
    xc = x.clone().requires_grad_(True)
    torch.relu(O.gcn_layer_ref(xc, adj, layer.weight.detach().cpu(), layer.bias.detach().cpu())).sum().backward()
    assert rel(xr.grad, xc.grad) < 1e-5


# ------------------------------------------------------------------------- GatedGCNStack
def _load_stack_from_golden(z, dtype):
    import ed_gated_gcn_b200 as E
    C, D2 = z["p_fc.0.weight"].shape
    D = D2 // 2
    stack = E.GatedGCNStack(D, n_layers=2, n_classes=C, gate_arch="sig-2", compute_dtype=dtype).to(DEV)
    sd = {k[2:]: torch.from_numpy(z[k]) for k in z if k.startswith("p_") and not k.startswith("p_dense.")}
    stack.load_state_dict(sd)                                        # same keys as BertAmir55 (bert_amir5.py:559-572)
    dense = torch.nn.Linear(z["p_dense.weight"].shape[1], C).to(DEV)
    with torch.no_grad():
        dense.weight.copy_(torch.from_numpy(z["p_dense.weight"]))
        dense.bias.copy_(torch.from_numpy(z["p_dense.bias"]))
    return stack, dense


def _oracle_params(stack, dense):
    sd = {k: v.detach().cpu().clone().requires_grad_(True) for k, v in stack.state_dict().items()}
    dw = dense.weight.detach().cpu().clone().requires_grad_(True)
    db = dense.bias.detach().cpu().clone().requires_grad_(True)
    lead, pairs = O.GATE_ARCHS[stack.gate_arch]
    off = 1 if lead else 0
    gcn_p = [(sd[f"gc{l}.weight"], sd[f"gc{l}.bias"]) for l in range(1, stack.n_layers + 1)]
    gate_p = [[(sd[f"gate{l}.{off + 2 * i}.weight"], sd[f"gate{l}.{off + 2 * i}.bias"]) for i in range(pairs)]
              for l in range(1, stack.n_layers + 1)]
    return sd, dw, db, gcn_p, gate_p, lead


def _oracle_run(stack, dense, sentences, targets, extra_feat=None, forced=None):
    """CPU oracle over a list of (x [T,D], adj [T,T], anchor, dist [T]) sentences sharing T or not;
    each sentence is one call of the reference block with batch 1, batch means re-assembled.
    forced = (final_arg [B,D], view_arg [V,B,D]) as sentence-local token indices."""
    sd, dw, db, gcn_p, gate_p, lead = _oracle_params(stack, dense)
    B = len(sentences)
    xs, logits, scores, xouts, views_vals, final_vals = [], [], [], [], [], []
    xy = kl = 0.0
    for b, (xb, adj, anc, d) in enumerate(sentences):
        xb = xb.clone().requires_grad_(True)
        feat = None if extra_feat is None else extra_feat[b:b + 1]

        def logits_fn(a, p):
            cat = [a, p] if feat is None else [feat, a, p]
            return torch.cat(cat, 1) @ dw.t() + db

        o = O.gated_block_ref(xb[None], adj[None], torch.tensor([anc]), d[None], gcn_p, gate_p,
                              sd["fc.0.weight"], sd["fc.0.bias"], logits_fn, lead_sigmoid=lead,
                              forced_view_arg=None if forced is None else forced[1][:, b:b + 1],
                              forced_final_arg=None if forced is None else forced[0][b:b + 1])
        xs.append(xb); logits.append(o["logits"]); scores.append(o["scores"][0]); xouts.append(o["x_out"][0])
        views_vals.append([(o["hs"][0][0] * g[0][None, :]).detach() for g in o["gates"]])
        final_vals.append(o["x_out"][0].detach())
        xy = xy + o["xy"] / B
        kl = kl + o["kl"] / B
    logits = torch.cat(logits)
    loss = torch.nn.functional.cross_entropy(logits, targets) + 0.01 * xy + 0.01 * kl      # train.py:115-118
    loss.backward()
    grads = {k: v.grad for k, v in sd.items()}
    grads["dense.weight"], grads["dense.bias"] = dw.grad, db.grad
    return dict(logits=logits, scores=scores, x_out=xouts, xy=xy, kl=kl, loss=loss, dx=[t.grad for t in xs],
                grads=grads, views_vals=views_vals, final_vals=final_vals)


def _local_args(out, sent_starts):
    """global arg-max rows of the CUDA path -> sentence-local token indices."""
    starts = torch.as_tensor(sent_starts, dtype=torch.int64)
    fa = out.pooled_arg.cpu().long() - starts[:, None]
    va = out.view_arg.cpu().long() - starts[None, :, None]
    return fa, va


def _check_routing(out, ora, sent_starts, max_frac=0.06, near=2e-2):
    """bf16 only: the CUDA path may pick another row than the fp32 reference ONLY where the two
    candidates tie within bf16 resolution; and that must be rare."""
    fa, va = _local_args(out, sent_starts)
    B, D = fa.shape
    n_flip = n_tot = 0
    for b in range(B):
        groups = [(ora["final_vals"][b], fa[b])] + [(ora["views_vals"][b][v], va[v, b]) for v in range(va.shape[0])]
        for vals, arg in groups:
            best, best_arg = vals.max(0)
            mine = vals.gather(0, arg[None, :])[0]
            flip = arg != best_arg
            n_flip += int(flip.sum()); n_tot += D
            scale = vals.abs().max(0)[0].clamp_min(1e-6)
            assert ((best - mine)[flip] <= near * scale[flip]).all(), "re-routed position is not a near-tie"
    assert n_flip <= max_frac * n_tot, (n_flip, n_tot)
    return fa, va


def _compare(out, loss, x_grad, stack, dense, ora, ora_grad, tol, L):
    assert rel(out.logits, ora["logits"]) < tol
    assert rel(out.scores.reshape(-1), torch.cat([s.reshape(-1) for s in ora["scores"]])) < tol
    if L > 1:
        assert rel(out.xy, ora["xy"]) < tol
    assert rel(out.kl, ora["kl"]) < tol
    assert rel(loss, ora["loss"]) < tol
    assert rel(x_grad.reshape(-1, x_grad.shape[-1]), torch.cat(ora_grad["dx"])) < tol, "dx"
    for name, p in list(stack.named_parameters()) + [("dense.weight", dense.weight), ("dense.bias", dense.bias)]:
        want = ora_grad["grads"][name]
        if name == "fc.0.bias" or want is None or want.abs().max() < 1e-9:
            continue                  # c_b cancels inside the softmax: that gradient is rounding noise
        assert rel(p.grad, want) < tol, name


@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "bf16"])
def test_stack_matches_full_reference_forward_backward(dtype):
    """BertAmir55.forward + backward as run by the reference (golden block55), dense-compat layout:
    every sentence has T rows, pad rows are live self-loop singletons (SURVEY fact 6)."""
    import ed_gated_gcn_b200 as E
    z = fixtures.load(os.path.join(GOLDEN, "block55.npz"))
    tol = tol_for(dtype)
    stack, dense = _load_stack_from_golden(z, dtype)
    x = torch.from_numpy(z["x"]).to(DEV).requires_grad_(True)          # LSTM output [B,T,D]
    adj = torch.from_numpy(z["adj"]).to(DEV)
    anchor = torch.from_numpy(z["anchor"]).to(DEV)
    dist = torch.from_numpy(z["dist"]).to(DEV)
    anchor_rep = torch.from_numpy(z["anchor_rep"]).to(DEV)
    targets = torch.from_numpy(z["targets"])
    graph = E.graph_from_dense(adj)
    B, T, D = x.shape

    def logits_fn(a, pooled):                                          # bert_amir5.py:643
        return dense(torch.cat([anchor_rep, a, pooled], dim=1))

    out = stack(x, graph, anchor, dist, logits_fn, head_params=list(dense.parameters()))
    loss = torch.nn.functional.cross_entropy(out.logits, targets.to(DEV)) + 0.01 * out.xy + 0.01 * out.kl
    loss.backward()
    # forward against the reference's own numbers
    for k in ("logits", "scores", "xy", "kl"):
        assert rel(getattr(out, k), z[k]) < tol, k
    assert rel(loss, z["loss"]) < tol
    if dtype == torch.float32:
        # backward against the reference's own numbers
        assert rel(x.grad, z["dx"]) < tol
        got = dict(stack.named_parameters())
        for k in z:
            if k.startswith("g_") and k != "g_fc.0.bias":
                name = k[2:]
                g = dense.weight.grad if name == "dense.weight" else dense.bias.grad if name == "dense.bias" \
                    else got[name].grad
                assert rel(fixtures.pick(z, k, g), z[k]) < tol, name
        return
    # bf16: gradients against the oracle (pinned to the same fixture) with the CUDA path's routing
    sents = [(torch.from_numpy(z["x"][b]), torch.from_numpy(z["adj"][b]), int(z["anchor"][b]),
              torch.from_numpy(z["dist"][b])) for b in range(B)]
    ora = _oracle_run(stack, dense, sents, targets, extra_feat=torch.from_numpy(z["anchor_rep"]))
    forced = _check_routing(out, ora, [b * T for b in range(B)], max_frac=0.08)
    ora_f = _oracle_run(stack, dense, sents, targets, extra_feat=torch.from_numpy(z["anchor_rep"]), forced=forced)
    _compare(out, loss, x.grad, stack, dense, ora, ora_f, tol, 2)


@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "bf16"])
@pytest.mark.parametrize("cfg", [dict(L=2, arch="sig-2", D=300, C=34, B=32, lo=5, hi=50),     # config C1
                                 dict(L=3, arch="3", D=64, C=7, B=9, lo=1, hi=20),
                                 dict(L=1, arch="2", D=32, C=2, B=5, lo=2, hi=9),
                                 dict(L=4, arch="sig-3", D=128, C=5, B=6, lo=30, hi=90),
                                 # config-4 shape: sentences too long for a shared-memory window (per-sentence / flat
                                 # kernels), D = 768 (streaming tcgen05 GEMM, 7 M tiles in wgrad), a hub of degree ~n/2
                                 dict(L=2, arch="sig-2", D=768, C=5, B=4, lo=200, hi=512, skewed=True),
                                 # config-3 shape: 768-d BERT-base features into a 3-layer gated stack, sentences <= 50 tokens
                                 dict(L=3, arch="sig-2", D=768, C=34, B=12, lo=5, hi=50)],
                         ids=["C1", "L3", "L1", "L4", "C4long", "C3"])
def test_stack_packed_rows_vs_oracle(dtype, cfg):
    """Packed layout (no pad rows): the oracle is run per sentence with T = n_b, which is the
    same convention (SURVEY hard part 2)."""
    import ed_gated_gcn_b200 as E
    from ed_gated_gcn_b200 import synth
    tol = tol_for(dtype)
    torch.manual_seed(1000 + cfg["D"] + cfg["L"])       # the head (nn.Linear) initialises from the global RNG
    batch = synth.make_batch(cfg["B"], cfg["lo"], cfg["hi"], seed=cfg["D"], skewed=cfg.get("skewed", False))
    D, C, B, Lyr = cfg["D"], cfg["C"], cfg["B"], cfg["L"]
    stack = E.GatedGCNStack(D, n_layers=Lyr, n_classes=C, gate_arch=cfg["arch"], compute_dtype=dtype).to(DEV)
    gen = torch.Generator().manual_seed(3)
    O.reference_init_([p for p in stack.parameters()], gen)            # train.py:75-84
    dense = torch.nn.Linear(2 * D, C).to(DEV)
    graph = E.build_graph(torch.from_numpy(batch.heads), torch.from_numpy(batch.sent_ptr), device=DEV)
    anchor = torch.from_numpy(batch.anchor).to(DEV)
    dist = E.tree_distance(graph, anchor)
    xp = torch.randn(batch.n_rows, D, generator=gen)
    targets = torch.arange(B) % C
    x = xp.to(DEV).requires_grad_(True)
    out = stack(x, graph, anchor, dist, lambda a, p: dense(torch.cat([a, p], 1)),
                head_params=list(dense.parameters()), return_x_out=True)
    loss = torch.nn.functional.cross_entropy(out.logits, targets.to(DEV)) + 0.01 * out.xy + 0.01 * out.kl
    loss.backward()

    sp = batch.sent_ptr
    sents = []
    for b, h in enumerate(batch.heads_list()):
        sents.append((xp[sp[b]:sp[b + 1]], torch.from_numpy(O.dense_adjacency_from_heads(h, len(h))).float(),
                      int(batch.anchor[b]), torch.tensor(O.tree_distance_bfs(h, int(batch.anchor[b])))))
    ora = _oracle_run(stack, dense, sents, targets)
    assert rel(out.x_out, torch.cat(ora["x_out"])) < tol
    ora_g = ora
    if dtype == torch.bfloat16:
        forced = _check_routing(out, ora, sp[:-1])
        ora_g = _oracle_run(stack, dense, sents, targets, forced=forced)
    _compare(out, loss, x.grad, stack, dense, ora, ora_g, tol, Lyr)


@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "bf16"])
def test_bert_amir54_variant_matches_full_reference_forward_backward(dtype):
    """BertAmir54.forward + backward as run by the reference (golden block54): fc = Sequential(Sigmoid, Linear)
    (bert_amir5.py:464-465), dense = two Linears over cat[aspect, out, pooled_output] (:443-446, :536)."""
    import ed_gated_gcn_b200 as E
    z = fixtures.load(os.path.join(GOLDEN, "block54.npz"))
    tol = tol_for(dtype)
    C, D2 = z["p_fc.1.weight"].shape
    D = D2 // 2
    stack = E.GatedGCNStack(D, n_layers=2, n_classes=C, gate_arch="sig-2", compute_dtype=dtype, fc_sigmoid=True).to(DEV)
    sd = {k[2:]: torch.from_numpy(z[k]) for k in z if k.startswith("p_") and not k.startswith("p_dense.")}
    stack.load_state_dict(sd)                                         # keys of BertAmir54 incl. fc.1.*
    dense = torch.nn.Sequential(torch.nn.Linear(2 * D + 768, 768), torch.nn.Linear(768, C)).to(DEV)
    dense.load_state_dict({k[len("p_dense."):]: torch.from_numpy(z[k]) for k in z if k.startswith("p_dense.")})
    x = torch.from_numpy(z["x"]).to(DEV).requires_grad_(True)
    adj = torch.from_numpy(z["adj"]).to(DEV)
    anchor = torch.from_numpy(z["anchor"]).to(DEV)
    dist = torch.from_numpy(z["dist"]).to(DEV)
    pooled_output = torch.from_numpy(z["dense_in"][:, 2 * D:]).to(DEV)
    targets = torch.from_numpy(z["targets"])
    graph = E.graph_from_dense(adj)
    out = stack(x, graph, anchor, dist, lambda a, p: dense(torch.cat([a, p, pooled_output], dim=1)),
                head_params=list(dense.parameters()))
    loss = torch.nn.functional.cross_entropy(out.logits, targets.to(DEV)) + 0.01 * out.xy + 0.01 * out.kl
    loss.backward()
    for k in ("logits", "scores", "xy", "kl"):
        assert rel(getattr(out, k), z[k]) < tol, k
    assert rel(loss, z["loss"]) < tol
    if dtype == torch.float32:
        assert rel(x.grad, z["dx"]) < tol
        got = dict(stack.named_parameters())
        got.update({"dense." + n: p for n, p in dense.named_parameters()})
        for k in z:
            if k.startswith("g_") and k not in ("g_fc.1.bias", "g_fc.1.weight"):
                assert rel(fixtures.pick(z, k, got[k[2:]].grad), z[k]) < tol, k
        # fc.1.weight: d kl / d fc.weight = sum_b sum_t ds_bt logits_b (x) sigmoid(cat[x_out_t, a_b]) with sum_t ds_bt = 0
        # (a softmax derivative): a 2.9e-6 remainder of summands that add up to 4.9e-4 in absolute value.  The
        # reference's OWN fp32 value is 1.6e-5 away from an fp64 evaluation of the same lines, i.e. outside the 1e-5
        # bar -- so this tensor is judged against fp64, with the error bound of the cancelling sum it is: a few dozen
        # fp32 roundings of the summands' magnitude (64 eps x sum |summand|), not 1e-5 of the remainder.
        g64, sum_abs = _fp64_fc_weight_grad_block54(z)
        bound = 64 * 1.1920929e-07 * sum_abs
        err = (got["fc.1.weight"].grad.detach().cpu().double() - g64).abs().max().item()
        err_ref = (torch.from_numpy(z["g_fc.1.weight"]).double() - g64).abs().max().item()
        assert err_ref < bound                                          # the reference's fp32 run obeys the same bound
        assert err < bound, (err, bound, err_ref)


@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "bf16"])
def test_bert_amir_variant_matches_full_reference_forward_backward(dtype):
    """BertAmir.forward + backward as run by the reference (golden bert_amir.npz): masked diversity pools
    (bert_amir.py:141-142), the trigger vector handed in (word-piece max-pool, :118), 3 x (Linear, Sigmoid) gates,
    fc a plain Linear, dense over cat[pooled_output, out] (:149)."""
    import ed_gated_gcn_b200 as E
    z = np.load(os.path.join(GOLDEN, "bert_amir.npz"))
    tol = tol_for(dtype)
    C, D2 = z["p_fc.weight"].shape
    D = D2 // 2
    stack = E.GatedGCNStack(D, n_layers=2, n_classes=C, gate_arch="3", compute_dtype=dtype).to(DEV)
    sd = {("fc.0." + k[5:] if k.startswith("p_fc.") else k[2:]): torch.from_numpy(z[k])
          for k in z.files if k.startswith("p_") and not k.startswith("p_dense.")}
    stack.load_state_dict(sd)                                         # gate{l}.{0,2,4}.*, gc{l}.*; fc.* -> fc.0.*
    dense = torch.nn.Linear(768 + D, C).to(DEV)
    dense.load_state_dict({k[len("p_dense."):]: torch.from_numpy(z[k]) for k in z.files if k.startswith("p_dense.")})
    x = torch.from_numpy(z["x"]).to(DEV).requires_grad_(True)
    aspect = torch.from_numpy(z["aspect"]).to(DEV).requires_grad_(True)
    adj = torch.from_numpy(z["adj"]).to(DEV)
    pooled_output = torch.from_numpy(z["pooled_output"]).to(DEV)
    view_len = torch.from_numpy((z["view_mask"] == 0).sum(1)).to(DEV)
    targets = torch.from_numpy(z["targets"])
    graph = E.graph_from_dense(adj)
    out = stack(x, graph, torch.from_numpy(z["anchor"]).to(DEV), torch.from_numpy(z["dist"]).to(DEV),
                lambda a, p: dense(torch.cat([pooled_output, p], dim=1)), head_params=list(dense.parameters()),
                aspect=aspect, view_len=view_len)
    loss = torch.nn.functional.cross_entropy(out.logits, targets.to(DEV)) + 0.01 * out.xy + 0.01 * out.kl
    loss.backward()
    for k in ("logits", "xy", "kl"):
        assert rel(getattr(out, k), z[k]) < tol, k
    assert rel(loss, z["loss"]) < tol
    if dtype == torch.float32:                    # (bf16: the routing rule of DESIGN 4 applies; the forward is pinned above)
        assert rel(x.grad, z["dx"]) < tol
        assert rel(aspect.grad, z["daspect"]) < tol
        got = {("fc." + n[5:] if n.startswith("fc.0.") else n): p for n, p in stack.named_parameters()}
        got.update({"dense." + n: p for n, p in dense.named_parameters()})
        for k in z.files:
            if k.startswith("g_") and k != "g_fc.bias":
                assert rel(got[k[2:]].grad, z[k]) < tol, k


def _fp64_fc_weight_grad_block54(z):
    """fp64 evaluation of the reference block on the block54 fixture (oracle restatement of bert_amir5.py:515-540 with
    fc = Sequential(Sigmoid, Linear)): d loss / d fc.1.weight and max_cj sum_bt |ds_bt logits_bc sigmoid(cat)_j|."""
    P = {k[2:]: torch.from_numpy(z[k]).double().requires_grad_(True) for k in z if k.startswith("p_")}
    D = z["x"].shape[2]
    x, adj = torch.from_numpy(z["x"]).double(), torch.from_numpy(z["adj"]).double()
    po = torch.from_numpy(z["dense_in"][:, 2 * D:]).double()
    gcn_p = [(P["gc1.weight"], P["gc1.bias"]), (P["gc2.weight"], P["gc2.bias"])]
    gate_p = [[(P[f"gate{l}.1.weight"], P[f"gate{l}.1.bias"]), (P[f"gate{l}.3.weight"], P[f"gate{l}.3.bias"])] for l in (1, 2)]
    fn = lambda a, p: (torch.cat([a, p, po], 1) @ P["dense.0.weight"].t() + P["dense.0.bias"]) @ P["dense.1.weight"].t() \
        + P["dense.1.bias"]
    o = O.gated_block_ref(x, adj, torch.from_numpy(z["anchor"]).long(), torch.from_numpy(z["dist"]).long(), gcn_p, gate_p,
                          P["fc.1.weight"], P["fc.1.bias"], fn, lead_sigmoid=True, fc_sigmoid=True)
    o["scores"].retain_grad()
    loss = torch.nn.functional.cross_entropy(o["logits"], torch.from_numpy(z["targets"]).long()) + 0.01 * o["xy"] + 0.01 * o["kl"]
    loss.backward()
    B, T, _ = x.shape
    cat = torch.sigmoid(torch.cat([o["x_out"].detach(), o["aspect"].detach()[:, None, :].expand(B, T, D)], 2))
    sum_abs = torch.einsum("bt,bc,btj->cj", o["scores"].grad.abs(), o["logits"].detach().abs(), cat).max().item()
    return P["fc.1.weight"].grad, sum_abs


def test_ungated_ablation_matches_oracle():
    """gated=False = BertAmir55NoGate (bert_amir5.py:654-760): same kernels with a unit gate, xy = 0.0, gate
    parameters present in the state dict (the reference constructs them, :672-681) but untouched by backward."""
    import ed_gated_gcn_b200 as E
    from ed_gated_gcn_b200 import synth
    torch.manual_seed(5)
    batch = synth.make_batch(11, 1, 30, seed=41)
    D, C, B = 48, 5, batch.n_graphs
    stack = E.GatedGCNStack(D, n_layers=2, n_classes=C, gated=False).to(DEV)
    gen = torch.Generator().manual_seed(6)
    O.reference_init_([p for p in stack.parameters()], gen)
    dense = torch.nn.Linear(2 * D, C).to(DEV)
    assert "gate1.1.weight" in stack.state_dict()
    graph = E.build_graph(torch.from_numpy(batch.heads), torch.from_numpy(batch.sent_ptr), device=DEV)
    anchor = torch.from_numpy(batch.anchor).to(DEV)
    dist = E.tree_distance(graph, anchor)
    xp = torch.randn(batch.n_rows, D, generator=gen)
    targets = torch.arange(B) % C
    x = xp.to(DEV).requires_grad_(True)
    out = stack(x, graph, anchor, dist, lambda a, p: dense(torch.cat([a, p], 1)), head_params=list(dense.parameters()),
                return_x_out=True)
    loss = torch.nn.functional.cross_entropy(out.logits, targets.to(DEV)) + 0.01 * out.xy + 0.01 * out.kl
    loss.backward()
    assert float(out.xy) == 0.0
    sd = {k: v.detach().cpu().clone().requires_grad_(True) for k, v in stack.state_dict().items()}
    dw, db = (t.detach().cpu().clone().requires_grad_(True) for t in (dense.weight, dense.bias))
    gcn_p = [(sd["gc1.weight"], sd["gc1.bias"]), (sd["gc2.weight"], sd["gc2.bias"])]
    sp = batch.sent_ptr
    xs, logits, kl, scores, xouts = [], [], 0.0, [], []
    for b, h in enumerate(batch.heads_list()):
        xb = xp[sp[b]:sp[b + 1]].clone().requires_grad_(True)
        adj = torch.from_numpy(O.dense_adjacency_from_heads(h, len(h))).float()
        d = torch.tensor(O.tree_distance_bfs(h, int(batch.anchor[b])))
        o = O.ungated_block_ref(xb[None], adj[None], torch.tensor([int(batch.anchor[b])]), d[None], gcn_p,
                                sd["fc.0.weight"], sd["fc.0.bias"], lambda a, p: torch.cat([a, p], 1) @ dw.t() + db)
        xs.append(xb); logits.append(o["logits"]); scores.append(o["scores"][0]); xouts.append(o["x_out"][0])
        kl = kl + o["kl"] / B
    want_loss = torch.nn.functional.cross_entropy(torch.cat(logits), targets) + 0.01 * kl
    want_loss.backward()
    assert rel(out.logits, torch.cat(logits)) < 1e-5 and rel(out.kl, kl) < 1e-5 and rel(loss, want_loss) < 1e-5
    assert rel(out.scores, torch.cat(scores)) < 1e-5 and rel(out.x_out, torch.cat(xouts)) < 1e-5
    assert rel(x.grad, torch.cat([t.grad for t in xs])) < 1e-5
    for name in ("gc1.weight", "gc1.bias", "gc2.weight", "gc2.bias", "fc.0.weight"):
        assert rel(dict(stack.named_parameters())[name].grad, sd[name].grad) < 1e-5, name
    assert rel(dense.weight.grad, dw.grad) < 1e-5
    for name, p in stack.named_parameters():
        if name.startswith("gate"):
            assert p.grad is None or float(p.grad.abs().max()) == 0.0


def _dropout_mask_numpy(seed: int, stream_id: int, p: float, n_rows: int, D: int) -> np.ndarray:
    """keep(t,d) / (1-p) of edg_dropout_rows, restated with numpy uint32 arithmetic (include/edgcn.h)."""
    M = np.uint64(0xFFFFFFFF)

    def mix32(x):
        x = x & M
        x ^= x >> np.uint64(16); x = (x * np.uint64(0x7feb352d)) & M
        x ^= x >> np.uint64(15); x = (x * np.uint64(0x846ca68b)) & M
        x ^= x >> np.uint64(16)
        return x

    klo = np.uint64((seed & 0xFFFFFFFF) ^ ((stream_id * 0xC2B2AE3D) & 0xFFFFFFFF))
    khi = np.uint64((seed >> 32) & 0xFFFFFFFF)
    rows = np.arange(n_rows, dtype=np.uint64)[:, None]
    cols = np.arange(D, dtype=np.uint64)[None, :]
    u = mix32(mix32((rows * np.uint64(0x9E3779B1) + klo) & M) ^ ((cols * np.uint64(0x85EBCA77) + khi) & M))
    thr = np.uint64(min(int(p * 4294967296.0), 4294967295))
    scale = np.float32(1.0) / (np.float32(1.0) - np.float32(p))
    return np.where(u >= thr, scale, np.float32(0.0)).astype(np.float32)


def test_dropout_rows_kernel_matches_the_numpy_restatement():
    from ed_gated_gcn_b200 import ops
    for dtype in DTYPES:
        x = ops.as_rows(torch.randn(97, 44).to(DEV), dtype)
        seed = torch.tensor([0x1234_5678_9ABC_DEF1 >> 1], dtype=torch.int64, device=DEV)
        y = ops.dropout_rows(x, seed, 3, 0.25)
        m = torch.from_numpy(_dropout_mask_numpy(int(seed), 3, 0.25, 97, 44))
        want = (x.float().cpu() * m)
        assert torch.equal(y.float().cpu(), want.to(dtype).float())
        assert 0.68 < float((m > 0).float().mean()) < 0.82
        base = y.as_strided((97, y.stride(0)), (y.stride(0), 1))
        assert (base[:, 44:] == 0).all()
        acc = ops.alloc_rows(97, 44, dtype, DEV, zero=True)
        acc.copy_(y)
        z = ops.dropout_rows(x, seed, 3, 0.25, out=acc, accumulate=True)
        assert rel(z.float().cpu(), 2 * want) < (1e-6 if dtype == torch.float32 else 8e-3)


@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "bf16"])
@pytest.mark.parametrize("Lyr", [2, 3])
def test_stack_training_mode_gate_dropout_vs_oracle(dtype, Lyr):
    """Training mode with dropout p = 0.25 (the reference default, train.py:294): nn.Dropout on the broadcast
    gates (bert_amir5.py:624-625).  The oracle gets the SAME masks, rebuilt with numpy from the seed the stack drew."""
    import ed_gated_gcn_b200 as E
    from ed_gated_gcn_b200 import synth
    tol = tol_for(dtype)
    torch.manual_seed(77 + Lyr)
    batch = synth.make_batch(10, 2, 24, seed=50 + Lyr)
    D, C, B, p = 40, 4, batch.n_graphs, 0.25
    stack = E.GatedGCNStack(D, n_layers=Lyr, n_classes=C, compute_dtype=dtype, dropout=p).to(DEV).train()
    gen = torch.Generator().manual_seed(8)
    O.reference_init_([q for q in stack.parameters()], gen)
    dense = torch.nn.Linear(2 * D, C).to(DEV)
    graph = E.build_graph(torch.from_numpy(batch.heads), torch.from_numpy(batch.sent_ptr), device=DEV)
    anchor = torch.from_numpy(batch.anchor).to(DEV)
    dist = E.tree_distance(graph, anchor)
    xp = torch.randn(batch.n_rows, D, generator=gen)
    targets = torch.arange(B) % C
    x = xp.to(DEV).requires_grad_(True)
    out = stack(x, graph, anchor, dist, lambda a, q: dense(torch.cat([a, q], 1)), head_params=list(dense.parameters()),
                return_x_out=True)
    loss = torch.nn.functional.cross_entropy(out.logits, targets.to(DEV)) + 0.01 * out.xy + 0.01 * out.kl
    loss.backward()
    seed = int(stack.last_dropout_seed)
    masks = [torch.from_numpy(_dropout_mask_numpy(seed, v, p, batch.n_rows, D)) for v in range(Lyr)]
    assert float((out.x_out == 0).float().mean()) > 0.15                  # dropped positions are really zero

    def run_oracle(forced=None):
        sd, dw, db, gcn_p, gate_p, lead = _oracle_params(stack, dense)
        sp = batch.sent_ptr
        xs, logits, scores, xouts, vv, fv = [], [], [], [], [], []
        xy = kl = 0.0
        for b, h in enumerate(batch.heads_list()):
            lo, hi = int(sp[b]), int(sp[b + 1])
            xb = xp[lo:hi].clone().requires_grad_(True)
            adj = torch.from_numpy(O.dense_adjacency_from_heads(h, len(h))).float()
            d = torch.tensor(O.tree_distance_bfs(h, int(batch.anchor[b])))
            o = O.gated_block_ref(xb[None], adj[None], torch.tensor([int(batch.anchor[b])]), d[None], gcn_p, gate_p,
                                  sd["fc.0.weight"], sd["fc.0.bias"], lambda a, q: torch.cat([a, q], 1) @ dw.t() + db,
                                  lead_sigmoid=lead, gate_masks=[m[lo:hi][None] for m in masks],
                                  forced_view_arg=None if forced is None else forced[1][:, b:b + 1],
                                  forced_final_arg=None if forced is None else forced[0][b:b + 1])
            xs.append(xb); logits.append(o["logits"]); scores.append(o["scores"][0]); xouts.append(o["x_out"][0])
            vv.append([(o["hs"][0][0] * g[0][None, :] * masks[i][lo:hi]).detach() for i, g in enumerate(o["gates"])])
            fv.append(o["x_out"][0].detach())
            xy = xy + o["xy"] / B
            kl = kl + o["kl"] / B
        lg = torch.cat(logits)
        ls = torch.nn.functional.cross_entropy(lg, targets) + 0.01 * xy + 0.01 * kl
        ls.backward()
        grads = {k: v.grad for k, v in sd.items()}
        grads["dense.weight"], grads["dense.bias"] = dw.grad, db.grad
        return dict(logits=lg, scores=scores, x_out=xouts, xy=xy, kl=kl, loss=ls, dx=[t.grad for t in xs], grads=grads,
                    views_vals=vv, final_vals=fv)

    ora = run_oracle()
    assert rel(out.x_out, torch.cat(ora["x_out"])) < tol
    ora_g = ora
    if dtype == torch.bfloat16:
        forced = _check_routing(out, ora, batch.sent_ptr[:-1], max_frac=0.2)   # many exact ties at the dropped zeros
        ora_g = run_oracle(forced)
    _compare(out, loss, x.grad, stack, dense, ora, ora_g, tol, Lyr)
    # eval mode = no dropout
    stack.eval()
    with torch.no_grad():
        out_e = stack(xp.to(DEV), graph, anchor, dist, lambda a, q: dense(torch.cat([a, q], 1)), return_x_out=True)
    assert float((out_e.x_out == 0).float().mean()) < 0.01
    # a trainable head that is not declared would train with a zero gradient: refused
    with pytest.raises(E.EdgError, match="head_params"):
        stack(xp.to(DEV), graph, anchor, dist, lambda a, q: dense(torch.cat([a, q], 1)))


def test_stack_rejects_cpu_tensors():
    import ed_gated_gcn_b200 as E
    from ed_gated_gcn_b200._lib import EdgError
    stack = E.GatedGCNStack(8, 2, 2, dropout=0.25)
    with pytest.raises(EdgError):
        stack(torch.zeros(3, 8), None, torch.zeros(1), torch.zeros(3), lambda a, p: a)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_tensors_on_a_second_gpu_with_device_0_current():
    """The reference selects its GPU with `--device cuda:N` and never calls set_device (train.py:286): tensors live on
    cuda:1 while device 0 is current.  Every launch must go to the tensors' device and its current stream, and the
    shared-memory opt-in of the kernels must happen per device."""
    import ed_gated_gcn_b200 as E
    from ed_gated_gcn_b200 import synth
    assert torch.cuda.current_device() == 0
    dev1 = torch.device("cuda", 1)
    batch = synth.make_batch(40, 3, 30, seed=12)
    D, C = 300, 5
    outs = []
    for dev in (torch.device("cuda", 0), dev1):
        torch.manual_seed(9)
        stack = E.GatedGCNStack(D, 2, C, compute_dtype="bf16").to(dev)
        dense = torch.nn.Linear(2 * D, C).to(dev)
        gen = torch.Generator().manual_seed(4)
        O.reference_init_(list(stack.parameters()) + list(dense.parameters()), gen)
        x = torch.randn(batch.n_rows, D, generator=gen).to(dev).requires_grad_(True)
        graph = E.build_graph(torch.from_numpy(batch.heads), torch.from_numpy(batch.sent_ptr), device=dev)
        anchor = torch.from_numpy(batch.anchor).to(dev)
        out = stack(x, graph, anchor, E.tree_distance(graph, anchor), lambda a, p: dense(torch.cat([a, p], 1)),
                    head_params=list(dense.parameters()))
        loss = out.logits.square().mean() + out.xy + out.kl
        loss.backward()
        torch.cuda.synchronize(dev)
        assert x.grad.device == dev
        outs.append((out.logits.detach().cpu(), float(out.kl), x.grad.cpu(), stack.gc1.weight.grad.cpu()))
        # the drop-in layer with a dense adjacency on that device as well
        layer = E.GraphConvolution(16, 16, None).to(dev)
        xs, adj, T = dense_inputs(synth.make_batch(5, 3, 9, seed=1), 16, seed=1)
        y = layer(xs.to(dev), adj.to(dev))
        assert rel(y, O.gcn_layer_ref(xs, adj, layer.weight.detach().cpu(), layer.bias.detach().cpu())) < 1e-5
    assert torch.cuda.current_device() == 0
    for a, b in zip(outs[0], outs[1]):              # same arithmetic on both devices: bitwise equal
        assert (torch.equal(a, b) if torch.is_tensor(a) else a == b)


@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "bf16"])
def test_dense_head_and_fused_loss_equal_the_torch_head(dtype):
    """`E.DenseHead` passed as logits_fn (run inside the block's head launches, edg_block_head_*) + `E.cross_entropy`
    against the same stack with torch's nn.Linear-on-cat head (the fc-only launches) and F.cross_entropy: same loss,
    same gradients everywhere."""
    import ed_gated_gcn_b200 as E
    from ed_gated_gcn_b200 import synth
    torch.manual_seed(5)
    D, C, B = 300, 34, 200
    batch = synth.make_batch(B, 5, 50, seed=3)
    stack = E.GatedGCNStack(D, n_layers=2, n_classes=C, gate_arch="sig-2", compute_dtype=dtype).to(DEV)
    head = E.DenseHead(2 * D, C).to(DEV)
    graph = E.build_graph(torch.from_numpy(batch.heads), torch.from_numpy(batch.sent_ptr), device=DEV)
    anchor = torch.from_numpy(batch.anchor).to(DEV)
    dist = E.tree_distance(graph, anchor)
    x = torch.randn(batch.n_rows, D, device=DEV).requires_grad_(True)
    tgt = (torch.arange(B) % C).to(DEV)
    params = list(stack.parameters()) + list(head.parameters())

    def run(fused):
        for p in params:
            p.grad = None
        x.grad = None
        if fused:
            out = stack(x, graph, anchor, dist, head)
            loss = E.cross_entropy(out.logits, tgt) + 0.01 * out.xy + 0.01 * out.kl
        else:
            out = stack(x, graph, anchor, dist, lambda a, p: torch.nn.functional.linear(torch.cat([a, p], 1), head.weight, head.bias),
                        head_params=list(head.parameters()))
            loss = torch.nn.functional.cross_entropy(out.logits, tgt) + 0.01 * out.xy + 0.01 * out.kl
        loss.backward()
        return out.logits.clone(), float(loss), [p.grad.clone() for p in params], x.grad.clone()

    torch.backends.cuda.matmul.allow_tf32 = False
    lg_t, loss_t, g_t, dx_t = run(False)
    lg_f, loss_f, g_f, dx_f = run(True)
    tol = 1e-5 if dtype == torch.float32 else 2e-3       # same bf16 kernels on both sides: only the head's fp32 rounding differs
    assert rel(lg_f, lg_t) < 1e-5
    assert abs(loss_f - loss_t) < 1e-5 * max(1.0, abs(loss_t))
    assert rel(dx_f, dx_t) < tol
    scale = max(float(b.abs().max()) for b in g_t)
    for a, b in zip(g_f, g_t):
        # against the larger of the tensor's own magnitude and 1e-3 of the largest gradient: fc.bias' gradient is
        # analytically zero here (1e-12 of rounding noise on both sides, next to gradients of 6e-2)
        assert a.shape == b.shape
        assert float((a - b).abs().max()) <= tol * max(float(b.abs().max()), 1e-3 * scale)
