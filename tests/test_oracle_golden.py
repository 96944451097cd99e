"""The oracle against the fixtures produced by the reference itself
(oracle/make_golden.py).  CPU only."""
import os

import numpy as np
import pytest
import torch

from oracle import fixtures, ref_oracle as O
from conftest import GOLDEN, rel_err


def test_gcn_layer_matches_reference_outputs():
    z = fixtures.load(os.path.join(GOLDEN, "gcn_layer.npz"))
    for ci in range(int(z["n_cases"])):
        p = f"c{ci}_"
        T = int(z[p + "T"])
        sp = z[p + "sent_ptr"]
        heads = [z[p + "heads"][sp[b]:sp[b + 1]] for b in range(len(sp) - 1)]
        adj = O.dense_batch_from_heads(heads, T)
        text = torch.tensor(z[p + "text"], requires_grad=True)
        w = torch.tensor(z[p + "weight"], requires_grad=True)
        b = torch.tensor(z[p + "bias"], requires_grad=True) if (p + "bias") in z else None
        y = O.gcn_layer_ref(text, adj, w, b)
        (y * torch.tensor(z[p + "probe"])).sum().backward()
        # same torch ops in the same order as models/gcn.py:33-45 -> bitwise equal
        assert torch.equal(y.detach(), torch.tensor(z[p + "y"]))
        assert rel_err(text.grad, z[p + "dtext"]) < 1e-6
        assert rel_err(w.grad, z[p + "dweight"]) < 1e-6
        if b is not None:
            assert rel_err(b.grad, z[p + "dbias"]) < 1e-6


def _cases():
    z = np.load(os.path.join(GOLDEN, "tree_dist.npz"))
    for i in range(len(z["target"])):
        lo, hi = z["ptr"][i], z["ptr"][i + 1]
        yield z["heads"][lo:hi], int(z["target"][i]), z["dist"][lo:hi], int(z["kind"][i])


def test_tree_distance_restatement_matches_reference_outputs():
    n = 0
    for heads, target, want, kind in _cases():
        adj = O.dense_adjacency_from_heads(heads, 100)
        got = O.tree_distance_ref(adj.tolist(), target, len(heads))
        assert got == [int(x) for x in want]
        n += 1
    assert n > 300


def test_bfs_and_forest_forms_match_reference_outputs():
    for heads, target, want, kind in _cases():
        if kind == 0:
            assert O.tree_distance_bfs(heads, target) == [int(x) for x in want]
        assert O.forest_distance(heads, target) == [int(x) for x in want]


def test_cycle_divergence_is_documented():
    """On a graph with a cycle the reference's walk over-estimates (SURVEY fact 8):
    ring of 6, trigger 0 -- node 5 is one hop away but the reference says 2 (+1)."""
    z = np.load(os.path.join(GOLDEN, "tree_dist_cycle.npz"))
    assert [int(x) for x in z["dist"]] == [1, 2, 3, 4, 5, 2]


def test_adjacency_is_identity_plus_symmetric_edges():
    m = O.dense_adjacency_from_edges([(1, 2), (2, 1), (3, 2)], 6)
    want = np.eye(6, dtype=np.int64)
    for i, j in ((0, 1), (1, 2)):
        want[i, j] = want[j, i] = 1
    assert (m == want).all()
    assert m[5, 5] == 1          # padding rows keep their self loop (graph.py:66)


def test_pad_rules():
    assert O.pad_distance([2, 1, 2], 5, "max+1") == [2, 1, 2, 3, 3]     # data_utils.py:486-488
    assert O.pad_distance([2, 1, 2], 5, "zero") == [2, 1, 2, 0, 0]      # data_utils.py:593-594


def test_block_matches_full_reference_forward_backward():
    z = fixtures.load(os.path.join(GOLDEN, "block55.npz"))
    P = {k[2:]: torch.tensor(z[k], requires_grad=True) for k in z if k.startswith("p_")}
    x = torch.tensor(z["x"], requires_grad=True)
    adj = torch.tensor(z["adj"])
    anchor = torch.tensor(z["anchor"], dtype=torch.long)
    dist = torch.tensor(z["dist"])
    anchor_rep = torch.tensor(z["anchor_rep"])

    def logits_fn(aspect, pooled):          # bert_amir5.py:643
        return torch.cat([anchor_rep, aspect, pooled], dim=1) @ P["dense.weight"].t() + P["dense.bias"]

    out = O.gated_block_ref(
        x, adj, anchor, dist,
        [(P["gc1.weight"], P["gc1.bias"]), (P["gc2.weight"], P["gc2.bias"])],
        [[(P["gate1.1.weight"], P["gate1.1.bias"]), (P["gate1.3.weight"], P["gate1.3.bias"])],
         [(P["gate2.1.weight"], P["gate2.1.bias"]), (P["gate2.3.weight"], P["gate2.3.bias"])]],
        P["fc.0.weight"], P["fc.0.bias"], logits_fn, lead_sigmoid=True)
    loss = O.block_loss_ref(out, torch.tensor(z["targets"]))
    loss.backward()
    tol = 2e-6
    assert rel_err(out["hs"][0], z["h1"]) < tol
    assert rel_err(out["hs"][1], z["h2"]) < tol
    assert rel_err(out["gates"][0], z["g1"]) < tol
    assert rel_err(out["gates"][1], z["g2"]) < tol
    for k in ("logits", "scores", "xy", "kl"):
        assert rel_err(out[k], z[k]) < tol, k
    assert rel_err(loss, z["loss"]) < tol
    assert rel_err(x.grad, z["dx"]) < 1e-5
    for name, p in P.items():
        if name == "fc.0.bias":      # c_b cancels inside the softmax (SURVEY A9): gradient is rounding noise
            assert p.grad.abs().max() < 1e-9 and np.abs(z["g_" + name]).max() < 1e-9
            continue
        assert rel_err(fixtures.pick(z, "g_" + name, p.grad), z["g_" + name]) < 1e-5, name


def test_bertdm_block_matches_reference_fixture(golden_dir):
    """N1 + N4 (SURVEY 8f): the restated word-piece bmm and BertDM left/right pooling reproduce the tensor the
    reference's own BertDM.forward feeds to its classifier, and its gradient, bit for bit."""
    z = np.load(os.path.join(golden_dir, "bertdm.npz"))
    transform, bert_x = torch.from_numpy(z["transform"]), torch.from_numpy(z["bert_x"]).requires_grad_(True)
    anchor, lengths = torch.from_numpy(z["anchor"]), torch.from_numpy(z["lengths"])
    x = O.wordpiece_bmm_ref(transform, bert_x)
    pooled = O.bertdm_pool_ref(x, anchor, lengths)
    anchor_rep = x[torch.arange(x.shape[0]), anchor]                    # bertdm.py:186-193 (masked_select)
    dense_in = torch.cat((anchor_rep, pooled), 1)
    assert torch.equal(dense_in, torch.from_numpy(z["dense_in"]))
    (dx,) = torch.autograd.grad(dense_in, bert_x, torch.from_numpy(z["probe"]))
    assert rel_err(dx, z["d_bert_x"]) < 1e-6
    # the transform the fixture was built with is the one data_utils.py:438-451 produces
    for b in range(transform.shape[0]):
        nz = (transform[b] != 0)
        assert nz.sum(1)[: int(lengths[b])].min() >= 1 and nz[int(lengths[b]):].sum() == 0


def test_block54_matches_full_reference_forward_backward():
    """BertAmir54 (fc = Sequential(Sigmoid, Linear), bert_amir5.py:464-465; two-layer dense head over
    cat[aspect, out, pooled_output], :443-446, :536) against the fixture produced by the reference's own forward."""
    z = fixtures.load(os.path.join(GOLDEN, "block54.npz"))
    P = {k[2:]: torch.tensor(z[k], requires_grad=True) for k in z if k.startswith("p_")}
    x = torch.tensor(z["x"], requires_grad=True)
    D = x.shape[-1]
    pooled_output = torch.tensor(z["dense_in"][:, 2 * D:])

    def logits_fn(aspect, pooled):          # bert_amir5.py:536
        h = torch.cat([aspect, pooled, pooled_output], dim=1) @ P["dense.0.weight"].t() + P["dense.0.bias"]
        return h @ P["dense.1.weight"].t() + P["dense.1.bias"]

    out = O.gated_block_ref(
        x, torch.tensor(z["adj"]), torch.tensor(z["anchor"], dtype=torch.long), torch.tensor(z["dist"]),
        [(P["gc1.weight"], P["gc1.bias"]), (P["gc2.weight"], P["gc2.bias"])],
        [[(P["gate1.1.weight"], P["gate1.1.bias"]), (P["gate1.3.weight"], P["gate1.3.bias"])],
         [(P["gate2.1.weight"], P["gate2.1.bias"]), (P["gate2.3.weight"], P["gate2.3.bias"])]],
        P["fc.1.weight"], P["fc.1.bias"], logits_fn, lead_sigmoid=True, fc_sigmoid=True)
    loss = O.block_loss_ref(out, torch.tensor(z["targets"]))
    loss.backward()
    for k in ("logits", "scores", "xy", "kl"):
        assert rel_err(out[k], z[k]) < 2e-6, k
    assert rel_err(loss, z["loss"]) < 2e-6
    assert rel_err(x.grad, z["dx"]) < 1e-5
    for name, p in P.items():
        if "g_" + name not in z or name == "fc.1.bias":
            continue
        if name == "fc.1.weight":
            # behind the Sigmoid the importance term's gradient is ~1e-6 in magnitude (its aspect half cancels inside
            # the softmax like the bias): summation-order noise of ~1e-11 is 1e-5 of that
            assert rel_err(p.grad, z["g_" + name]) < 1e-4, name
            continue
        assert rel_err(fixtures.pick(z, "g_" + name, p.grad), z["g_" + name]) < 1e-5, name


def test_bert_amir_block_matches_full_reference_forward_backward():
    """BertAmir (models/bert_amir.py:83-156): masked diversity pools (``masked_fill(mask, -1e12)``, :141-142), the
    word-piece-pooled trigger vector (:118), 3 x (Linear, Sigmoid) gates without a leading Sigmoid (:31-36), ``fc`` a
    plain Linear (:38), ``dense`` over cat[pooled_output, out] (:149) -- against the reference's own forward + backward."""
    z = np.load(os.path.join(GOLDEN, "bert_amir.npz"))
    P = {k[2:]: torch.tensor(z[k], requires_grad=True) for k in z.files if k.startswith("p_")}
    x = torch.tensor(z["x"], requires_grad=True)
    aspect = torch.tensor(z["aspect"], requires_grad=True)
    pooled_output = torch.tensor(z["pooled_output"])
    assert z["view_mask"].sum() > 0                      # the mask removes rows inside the padded length
    logits_fn = lambda a, pooled: torch.cat([pooled_output, pooled], dim=1) @ P["dense.weight"].t() + P["dense.bias"]
    out = O.gated_block_ref(
        x, torch.tensor(z["adj"]), torch.tensor(z["anchor"], dtype=torch.long), torch.tensor(z["dist"]),
        [(P["gc1.weight"], P["gc1.bias"]), (P["gc2.weight"], P["gc2.bias"])],
        [[(P[f"gate{l}.{i}.weight"], P[f"gate{l}.{i}.bias"]) for i in (0, 2, 4)] for l in (1, 2)],
        P["fc.weight"], P["fc.bias"], logits_fn, lead_sigmoid=False, aspect=aspect, view_mask=torch.tensor(z["view_mask"]))
    loss = O.block_loss_ref(out, torch.tensor(z["targets"]))
    loss.backward()
    for k in ("logits", "xy", "kl"):
        assert rel_err(out[k], z[k]) < 2e-6, k
    assert rel_err(loss, z["loss"]) < 2e-6
    assert rel_err(x.grad, z["dx"]) < 1e-5
    assert rel_err(aspect.grad, z["daspect"]) < 1e-5
    for name, p in P.items():
        if name == "fc.bias":
            continue
        assert rel_err(p.grad, z["g_" + name]) < 1e-5, name
