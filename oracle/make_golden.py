"""Generate the committed golden fixtures under ``tests/golden/`` by RUNNING THE
REFERENCE ITSELF (``/root/reference``, read-only, build container only).

The reference does not import as shipped (SURVEY.md fact 4): ``models/gcn.py``
imports a ``layers`` package that is not in the repository, ``data_utils.py``
imports spacy / pytorch_pretrained_bert.  None of those names is used on the hot
path, so empty stand-in modules are registered in ``sys.modules`` first; the
reference's own source files are then imported unmodified:

* ``models.gcn.GraphConvolution``            (models/gcn.py:9-45)
* ``data_utils.get_dist_to_target``          (data_utils.py:302-323)
* ``models.bert_amir5.BertAmir55``           (models/bert_amir5.py:544-650) with a stub
  BERT that returns seeded random layers, so the WHOLE reference forward
  (transform bmm, LSTM, gates, gc1, gc2, pooling, dense, fc, softmaxes) and its
  autograd backward run; the tensors entering and leaving the gated block are
  captured with hooks.

Run:  python oracle/make_golden.py        (writes tests/golden/*.npz, see oracle/fixtures.py)
This script is test infrastructure; it cannot run on the GPU box (no reference
there) -- which is why its outputs are committed.
"""
from __future__ import annotations

import os
import sys
import types

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get("EDG_REFERENCE", "/root/reference")
GOLD = os.path.join(ROOT, "tests", "golden")
sys.path.insert(0, ROOT)


def _install_stubs() -> None:
    def mod(name, **attrs):
        m = types.ModuleType(name)
        for k, v in attrs.items():
            setattr(m, k, v)
        sys.modules[name] = m
        return m

    class _Missing:  # any accidental use must fail loudly
        def __init__(self, *a, **k):
            raise RuntimeError("stub of a dependency the hot path never touches")

    mod("layers")
    mod("layers.squeeze_embedding", SqueezeEmbedding=_Missing)
    class _LstmStandIn(torch.nn.Module):
        """Stands for layers/dynamic_rnn.py (not in the repository): an LSTM over the padded batch; the lengths are
        ignored.  Only BertAmir / BertAmir2 use it, upstream of the block whose input the fixture captures."""
        def __init__(self, input_size, hidden_size, num_layers=1, batch_first=True, bidirectional=False, **kw):
            super().__init__()
            self.rnn = torch.nn.LSTM(input_size, hidden_size, num_layers=num_layers, batch_first=batch_first,
                                     bidirectional=bidirectional)

        def forward(self, x, x_len):
            return self.rnn(x)

    mod("layers.dynamic_rnn", DynamicLSTM=_LstmStandIn)
    mod("spacy")
    mod("pytorch_pretrained_bert", BertTokenizer=_Missing, BertModel=_Missing)
    sys.path.insert(0, REF)


def golden_gcn_layer(GraphConvolution) -> None:
    from ed_gated_gcn_b200 import synth
    from oracle import fixtures, ref_oracle as O
    out, drawn = {}, {}
    cases = [(3, 9, 16, 16, True, 0), (2, 50, 300, 300, True, 1), (4, 12, 24, 40, False, 2)]
    for ci, (B, T, Din, Dout, bias, seed) in enumerate(cases):
        g = torch.Generator().manual_seed(100 + seed)
        batch = synth.make_batch(B, max(2, T // 2), T, seed=seed + 7)
        adj = O.dense_batch_from_heads(batch.heads_list(), T)       # identity on pad rows too
        layer = GraphConvolution(Din, Dout, None, bias=bias)
        O.reference_init_(list(layer.parameters()), g)
        text = torch.randn(B, T, Din, generator=g, requires_grad=True)
        probe = torch.randn(B, T, Dout, generator=g)
        y = layer(text, adj)
        (y * probe).sum().backward()
        pre = f"c{ci}_"
        out[pre + "heads"] = batch.heads
        out[pre + "sent_ptr"] = batch.sent_ptr
        out[pre + "T"] = np.int64(T)
        out[pre + "text"] = text.detach().numpy()
        out[pre + "weight"] = layer.weight.detach().numpy()
        drawn[pre + "weight"] = (100 + seed, 0)                     # the first draws of g, bias next (reference_init_)
        if bias:
            out[pre + "bias"] = layer.bias.detach().numpy()
            out[pre + "dbias"] = layer.bias.grad.numpy()
            drawn[pre + "bias"] = (100 + seed, Din * Dout)
        out[pre + "probe"] = probe.numpy()
        out[pre + "y"] = y.detach().numpy()
        out[pre + "dtext"] = text.grad.numpy()
        out[pre + "dweight"] = layer.weight.grad.numpy()
    out["n_cases"] = np.int64(len(cases))
    fixtures.save(os.path.join(GOLD, "gcn_layer.npz"), out, drawn=drawn)
    print("gcn_layer.npz", len(out))


def golden_tree_dist(get_dist_to_target) -> None:
    from ed_gated_gcn_b200 import synth
    from oracle import ref_oracle as O
    rng = np.random.default_rng(14181)
    heads_cat, ptr, targets, dist_cat = [], [0], [], []
    kinds = []

    def add(heads, target, kind):
        n = len(heads)
        adj = O.dense_adjacency_from_heads(heads, 100)       # ORI_ML = 100, graph.py:42,66
        d = get_dist_to_target(adj.tolist(), int(target), [-1] * n, n)
        heads_cat.extend(int(h) for h in heads)
        ptr.append(len(heads_cat))
        targets.append(int(target))
        dist_cat.extend(int(x) for x in d)
        kinds.append(kind)

    # every target of a few small trees, then random (tree, target) pairs up to 64 tokens
    for n in (1, 2, 3, 5, 8, 13):
        for _ in range(3):
            h = synth.random_tree(n, rng)
            for t in range(n):
                add(h, t, 0)
    for _ in range(160):
        n = int(rng.integers(2, 65))
        h = synth.random_tree(n, rng, skewed=bool(rng.integers(0, 2)))
        add(h, int(rng.integers(0, n)), 0)
    # forests: cut 1-3 edges so some tokens cannot reach the trigger (data_utils.py:311)
    for _ in range(60):
        n = int(rng.integers(2, 40))
        h = synth.random_tree(n, rng).copy()
        kids = np.nonzero(h >= 0)[0]
        for c in rng.choice(kids, size=min(len(kids), int(rng.integers(1, 4))), replace=False):
            h[c] = -1
        add(h, int(rng.integers(0, n)), 1)
    np.savez_compressed(os.path.join(GOLD, "tree_dist.npz"),
                        heads=np.asarray(heads_cat, dtype=np.int32), ptr=np.asarray(ptr, dtype=np.int32),
                        target=np.asarray(targets, dtype=np.int32), dist=np.asarray(dist_cat, dtype=np.int64),
                        kind=np.asarray(kinds, dtype=np.int32))
    print("tree_dist.npz", len(targets), "cases")

    # one non-tree (a cycle): the reference's walk is order dependent there (SURVEY fact 8);
    # kept as documentation of the divergence, not as a parity target.
    h = np.array([-1, 0, 1, 2, 3, 4], dtype=np.int32)
    adj = O.dense_adjacency_from_heads(h, 100)
    adj[0, 5] = adj[5, 0] = 1
    d = get_dist_to_target(adj.tolist(), 0, [-1] * 6, 6)
    np.savez_compressed(os.path.join(GOLD, "tree_dist_cycle.npz"), heads=h, extra=np.array([0, 5]),
                        target=np.int32(0), dist=np.asarray(d, dtype=np.int64))
    print("tree_dist_cycle.npz", d)


def golden_block55(BertAmir55, fname: str = "block55.npz", seed: int = 55) -> None:
    """Also used for BertAmir54 (``block54.npz``): same inputs / hooks, the class differs in ``fc`` (a Sigmoid in
    front of the Linear, bert_amir5.py:464-465) and in the ``dense`` head (two Linears over cat[aspect, out,
    pooled_output], :443-446, :536)."""
    from ed_gated_gcn_b200 import synth
    from oracle import fixtures, ref_oracle as O
    torch.manual_seed(seed)
    B, ORI_ML, BERT_ML, C = 6, 20, 24, 5
    batch = synth.make_batch(B, 4, 14, seed=55)
    T = int(batch.lengths.max())

    class StubBert(torch.nn.Module):
        """Stands for the frozen BERT (train.py:43-44): 12 seeded random layers."""
        def forward(self, ids, seg, output_all_encoded_layers=True):
            g = torch.Generator().manual_seed(7)
            Bb, Lb = ids.shape
            layers = [torch.randn(Bb, Lb, 768, generator=g) * 0.5 for _ in range(12)]
            return layers, torch.randn(Bb, 768, generator=g)

    opt = types.SimpleNamespace(device="cpu", dropout=0.0, polarities_dim=C)
    model = BertAmir55(StubBert(), opt)
    g = torch.Generator().manual_seed(555)
    O.reference_init_([p for n, p in model.named_parameters()], g)      # train.py:75-84
    model.train()

    # inputs as data_utils.py / collate_fn lay them out
    bert_len = np.array([int(n) + 2 for n in batch.lengths])           # [CLS] w.. [SEP], one piece per word
    transform = np.zeros((B, ORI_ML, BERT_ML), dtype=np.float32)
    for b in range(B):
        for i in range(int(batch.lengths[b])):
            transform[b, i, i + 1] = 1.0                               # data_utils.py:438-451 with l = 1
    adj = np.stack([O.dense_adjacency_from_heads(h, ORI_ML) for h in batch.heads_list()]).astype(np.float32)
    dist = []
    for b, h in enumerate(batch.heads_list()):
        d = O.tree_distance_bfs(h, int(batch.anchor[b]))
        dist.append(O.pad_distance(d, ORI_ML, "max+1"))               # data_utils.py:486-488
    inputs = {
        "sentence_length": torch.tensor(batch.lengths, dtype=torch.long),
        "cls_text_sep_length": torch.tensor(bert_len, dtype=torch.long),
        "cls_text_sep_indices": torch.zeros(B, BERT_ML, dtype=torch.long),
        "cls_text_sep_segments_ids": torch.zeros(B, BERT_ML, dtype=torch.long),
        "transform": torch.tensor(transform),
        "anchor_index": torch.tensor(batch.anchor, dtype=torch.long),
        "dist_to_target": torch.tensor(dist, dtype=torch.long),
        "dependency_graph": torch.tensor(adj),
    }
    targets = torch.tensor(np.arange(B) % C, dtype=torch.long)

    cap = {}

    def lstm_hook(mod, inp, out):
        out[0].retain_grad()
        cap["x"] = out[0]

    def dense_pre(mod, inp):
        inp[0].retain_grad()
        cap["dense_in"] = inp[0]

    def gc_hook(name):
        def f(mod, inp, out):
            cap[name] = out
        return f

    model.lstm.register_forward_hook(lstm_hook)
    model.dense.register_forward_pre_hook(dense_pre)
    model.gc1.register_forward_hook(gc_hook("h1"))
    model.gc2.register_forward_hook(gc_hook("h2"))
    model.gate1.register_forward_hook(gc_hook("g1"))
    model.gate2.register_forward_hook(gc_hook("g2"))

    logits, xy, kl, scores = model(inputs)                              # bert_amir5.py:574-650
    loss = torch.nn.functional.cross_entropy(logits, targets) + 0.01 * xy + 0.01 * kl   # train.py:115-118
    loss.backward()

    out = {
        "heads": batch.heads, "sent_ptr": batch.sent_ptr, "anchor": batch.anchor, "T": np.int64(T),
        "targets": targets.numpy(),
        "x": cap["x"].detach().numpy(), "dx": cap["x"].grad.numpy(),
        "adj": adj[:, :T, :T], "dist": np.asarray(dist, dtype=np.int64)[:, :T],
        "anchor_rep": cap["dense_in"].detach().numpy()[:, :768 * 12],
        "dense_in": cap["dense_in"].detach().numpy(),
        "h1": cap["h1"].detach().numpy(), "h2": cap["h2"].detach().numpy(),
        "g1": cap["g1"].detach().numpy(), "g2": cap["g2"].detach().numpy(),
        "logits": logits.detach().numpy(), "xy": xy.detach().numpy(), "kl": kl.detach().numpy(),
        "scores": scores.detach().numpy(), "loss": loss.detach().numpy(),
    }
    keep = ("gc1.", "gc2.", "gate1.", "gate2.", "fc.", "dense.")
    drawn, offset = {}, 0
    for n, p in model.named_parameters():
        if n.startswith(keep):
            out["p_" + n] = p.detach().numpy()
            drawn["p_" + n] = (555, offset)                            # its place in the stream of g above
            if p.numel() < 500_000:                                    # BertAmir54's dense.0.weight is 768 x 1280: keep the
                out["g_" + n] = p.grad.numpy()                         # fixture small, its bias gradient pins that layer
        offset += p.numel()
    if fname != "block55.npz":
        out.pop("anchor_rep")
    else:
        out.pop("dense_in")                                            # block55.npz keeps its committed layout
    fixtures.save(os.path.join(GOLD, fname), out, drawn=drawn, sampled=[k for k in out if k.startswith("g_")])
    print(fname, {k: v.shape for k, v in out.items() if k[:2] not in ("p_", "g_")})


def golden_bertdm(BertDM) -> None:
    """The WHOLE ``BertDM.forward`` (models/bertdm.py:142-199) with a stub BERT: transform bmm, get_mask, left/right
    pooling, trigger-row gather.  The tensor entering ``self.dense`` (= cat[anchor_rep, pooledL-1, pooledR-1] in
    eval mode) is captured with a pre-hook, and its gradient w.r.t. the BERT output for a probe direction."""
    from oracle import ref_oracle as O
    rng = np.random.default_rng(77)
    g = torch.Generator().manual_seed(77)
    B, D = 7, 768                                    # bertdm.py:190 hard-codes 768 * n_layer
    lengths = np.array([9, 1, 12, 5, 12, 3, 7])
    anchor = np.array([0, 0, 11, 2, 5, 2, 6])        # first / last / interior triggers
    pieces = [rng.integers(1, 4, size=n).tolist() for n in lengths]
    transform = torch.FloatTensor([O.wordpiece_transform_ref(p) for p in pieces])        # collate_fn, data_utils.py:371
    bert_len = torch.LongTensor([sum(p) + 2 for p in pieces])                             # [CLS] + pieces + [SEP]
    Lmax = int(bert_len.max())
    bert_x = torch.randn(B, Lmax, D, generator=g)
    bert_x[3, 2:4] = -1.5 - bert_x[3, 2:4].abs()     # a left span that is negative everywhere: the masked zero wins
    bert_x.requires_grad_(True)

    class StubBert(torch.nn.Module):
        def forward(self, ids, seg, output_all_encoded_layers=True):
            return [bert_x], torch.zeros(B, D)

    opt = types.SimpleNamespace(device="cpu", n_layer=1, dropout=0.25, bert_dim=768, polarities_dim=5)
    model = BertDM(StubBert(), opt).eval()
    cap = {}
    model.dense.register_forward_pre_hook(lambda mod, inp: cap.__setitem__("dense_in", inp[0]))
    inputs = {"cls_text_sep_length": bert_len, "sentence_length": torch.LongTensor(lengths),
              "cls_text_sep_indices": torch.zeros(B, 120, dtype=torch.long),
              "cls_text_sep_segments_ids": torch.zeros(B, 120, dtype=torch.long),
              "anchor_index": torch.LongTensor(anchor), "transform": transform}
    model(inputs)
    probe = torch.randn(B, 3 * D, generator=g)
    (dx,) = torch.autograd.grad(cap["dense_in"], bert_x, probe)
    out = dict(transform=transform.numpy()[:, :int(lengths.max()), :Lmax], bert_x=bert_x.detach().numpy(),
               lengths=lengths, anchor=anchor, bert_len=bert_len.numpy(), dense_in=cap["dense_in"].detach().numpy(),
               probe=probe.numpy(), d_bert_x=dx.numpy())
    np.savez_compressed(os.path.join(GOLD, "bertdm.npz"), **out)
    print("bertdm.npz", {k: v.shape for k, v in out.items()})


def golden_bert_amir(BertAmir) -> None:
    """The WHOLE ``BertAmir.forward`` + backward (models/bert_amir.py:83-156) with a stub BERT and a stand-in for the
    absent ``layers.dynamic_rnn.DynamicLSTM`` (an nn.LSTM that ignores the lengths: the LSTM is upstream of the block,
    its output is captured as the block's input).  What the fixture pins: the masked diversity pools
    (``masked_fill(mask, -1e12)``, :141-142), the word-piece-pooled trigger vector (:118) feeding the 3 x (Linear,
    Sigmoid) gates (:31-36), ``fc`` as a plain Linear (:38) and the ``dense`` head over cat[pooled_output, out] (:149)."""
    from ed_gated_gcn_b200 import synth
    from oracle import ref_oracle as O
    torch.manual_seed(31)
    B, ORI_ML, BERT_ML, C, H = 6, 20, 30, 5, 32
    batch = synth.make_batch(B, 4, 14, seed=31)
    T = int(batch.lengths.max())
    rng = np.random.default_rng(31)
    pieces = [rng.integers(1, 3, size=int(n)).tolist() for n in batch.lengths]        # word pieces per word

    class StubBert(torch.nn.Module):
        def forward(self, ids, seg, output_all_encoded_layers=True):
            g = torch.Generator().manual_seed(9)
            Bb, Lb = ids.shape
            return [torch.randn(Bb, Lb, 768, generator=g) * 0.5 for _ in range(12)], torch.randn(Bb, 768, generator=g)

    opt = types.SimpleNamespace(device="cpu", dropout=0.0, polarities_dim=C, n_layer=1, bert_dim=768, hidden_dim=H)
    model = BertAmir(StubBert(), opt)
    g = torch.Generator().manual_seed(313)
    O.reference_init_([p for n, p in model.named_parameters()], g)      # train.py:75-84
    model.train()

    # inputs as data_utils.py:455-505 lays them out: [CLS] pieces [SEP] trigger pieces [SEP]
    transform = np.zeros((B, ORI_ML, BERT_ML), dtype=np.float32)
    aspect_mask = np.ones((B, BERT_ML), dtype=np.float32)
    cls_mask = np.ones((B, BERT_ML), dtype=np.float32)
    cls_len = np.zeros(B, dtype=np.int64)
    for b in range(B):
        tr = O.wordpiece_transform_ref(pieces[b], ORI_ML, BERT_ML)
        transform[b] = np.asarray(tr, dtype=np.float32)
        starts = 1 + np.concatenate([[0], np.cumsum(pieces[b])[:-1]])
        a0, al = int(starts[batch.anchor[b]]), int(pieces[b][batch.anchor[b]])
        aspect_mask[b, a0:a0 + al] = 0.0                                  # data_utils.py:470-472
        cls_len[b] = 1 + sum(pieces[b]) + 1 + al + 1
        cls_mask[b, :cls_len[b]] = 0.0                                    # data_utils.py:463-464
    # make the mask bite: shorten one sentence's unmasked prefix below the padded length T (the reference's mask is
    # indexed by WORD position but built from the WORD-PIECE length, so it only ever removes pad rows)
    adj = np.stack([O.dense_adjacency_from_heads(h, ORI_ML) for h in batch.heads_list()]).astype(np.float32)
    dist = [O.pad_distance(O.tree_distance_bfs(h, int(batch.anchor[b])), ORI_ML, "max+1") for b, h in enumerate(batch.heads_list())]
    inputs = {
        "sentence_length": torch.tensor(batch.lengths, dtype=torch.long),
        "cls_text_sep_aspect_sep_length": torch.tensor(cls_len, dtype=torch.long),
        "cls_text_sep_aspect_sep_indices": torch.zeros(B, BERT_ML, dtype=torch.long),
        "cls_text_sep_aspect_sep_segments_ids": torch.zeros(B, BERT_ML, dtype=torch.long),
        "cls_text_sep_aspect_sep_aspect_mask": torch.tensor(aspect_mask),
        "cls_text_sep_aspect_sep_mask": torch.tensor(cls_mask),
        "transform": torch.tensor(transform),
        "anchor_index": torch.tensor(batch.anchor, dtype=torch.long),
        "dist_to_target": torch.tensor(dist, dtype=torch.long),
        "dependency_graph": torch.tensor(adj),
    }
    targets = torch.tensor(np.arange(B) % C, dtype=torch.long)
    cap = {}

    def gate_pre(mod, inp):
        if "aspect" not in cap:
            inp[0].retain_grad()
            cap["aspect"] = inp[0]

    def gc1_pre(mod, inp):
        inp[0].retain_grad()
        cap["x"] = inp[0]

    model.gate1.register_forward_pre_hook(gate_pre)
    model.gc1.register_forward_pre_hook(gc1_pre)
    model.text_lstm.register_forward_hook(lambda mod, inp, outp: cap.__setitem__("x_lstm", outp[0]))
    model.dense.register_forward_pre_hook(lambda mod, inp: cap.__setitem__("dense_in", inp[0]))
    logits, xy, kl = model(inputs)                                       # bert_amir.py:83-156
    loss = torch.nn.functional.cross_entropy(logits, targets) + 0.01 * xy + 0.01 * kl
    loss.backward()
    L = int(cls_len.max())
    out = {
        "heads": batch.heads, "sent_ptr": batch.sent_ptr, "anchor": batch.anchor, "T": np.int64(T), "targets": targets.numpy(),
        "x": cap["x"].detach().numpy(), "dx": cap["x"].grad.numpy(),
        "aspect": cap["aspect"].detach().numpy(), "daspect": cap["aspect"].grad.numpy(),
        "x_lstm": cap["x_lstm"].detach().numpy(), "aspect_mask": aspect_mask[:, :L],
        "adj": adj[:, :T, :T], "dist": np.asarray(dist, dtype=np.int64)[:, :T], "view_mask": cls_mask[:, :T],
        "pooled_output": cap["dense_in"].detach().numpy()[:, :768],
        "logits": logits.detach().numpy(), "xy": xy.detach().numpy(), "kl": kl.detach().numpy(), "loss": loss.detach().numpy(),
    }
    for n, p in model.named_parameters():
        if n.startswith(("gc1.", "gc2.", "gate1.", "gate2.", "fc.", "dense.")):
            out["p_" + n] = p.detach().numpy()
            out["g_" + n] = p.grad.numpy()
    np.savez_compressed(os.path.join(GOLD, "bert_amir.npz"), **out)
    print("bert_amir.npz", {k: v.shape for k, v in out.items() if k[:2] not in ("p_", "g_")},
          "masked positions inside T:", int(cls_mask[:, :T].sum()))


def main() -> None:
    os.makedirs(GOLD, exist_ok=True)
    _install_stubs()
    from models.gcn import GraphConvolution            # reference, unmodified
    import data_utils                                  # reference, unmodified
    from models.bert_amir5 import BertAmir55           # reference, unmodified
    golden_gcn_layer(GraphConvolution)
    golden_tree_dist(data_utils.get_dist_to_target)
    golden_block55(BertAmir55)
    from models.bert_amir5 import BertAmir54           # reference, unmodified
    golden_block55(BertAmir54, "block54.npz", seed=54)
    from models.bertdm import BertDM                   # reference, unmodified
    golden_bertdm(BertDM)
    from models.bert_amir import BertAmir              # reference, unmodified (DynamicLSTM: stand-in below)
    golden_bert_amir(BertAmir)


if __name__ == "__main__":
    main()
