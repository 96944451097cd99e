"""BertDM's left/right pooling on grouped (sentence, trigger) pairs: ``lr_pool(h, graph, anchor, pairs=)``.

The references are the expanded batch (each sentence's rows copied once per pair, run through the per-sentence
``lr_pool``), ``oracle.bertdm_pool_ref`` on the padded ``[P, T, D]`` copy, and the reference's own BertDM fixture
(tests/golden/bertdm.npz).  Layouts come from the gated pairs tests, plus two of this file: anchors in no particular
order, and sentences outside the forward's shared-memory plan (more than 512 rows, more than 2048 pairs)."""
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN
from gpu_util import DEV, rel
from oracle import ref_oracle as O
from test_gpu_j_pairs import _expand, _graph, _layout, _lengths_batch

pytestmark = pytest.mark.gpu

LAYOUTS = ["mixed", "windows", "long", "extra", "512", "shuffled", "outside-plan"]


def _ptr(per):
    pp = np.zeros(len(per) + 1, dtype=np.int32)
    pp[1:] = np.cumsum([len(p) for p in per])
    return pp, np.asarray([a for p in per for a in p], dtype=np.int32)


def _layout_m(name):
    """(TreeBatch, pair_ptr, anchor): the gated pairs layouts and two of this file."""
    rng = np.random.default_rng(7)
    if name == "shuffled":
        # every token a candidate in a random order, repeated anchors, sentences without pairs, 1-token sentences
        L = [9, 1, 0, 40, 17, 1, 25, 3]
        b = _lengths_batch(L, seed=8)
        per = [list(rng.permutation(n)) + list(rng.integers(0, max(n, 1), size=n // 2)) if n and s != 4 else []
               for s, n in enumerate(L)]
        return (b,) + _ptr(per)
    if name == "outside-plan":
        # 600 rows, and 2100 pairs on 20 rows: both take the per-pair scan, next to sentences that do not
        L = [600, 20, 13, 0, 31]
        b = _lengths_batch(L, seed=9)
        per = [[599, 0, 300, 17, 300], list(rng.integers(0, 20, size=2100)), list(range(13))[::-1], [], [30, 0, 15]]
        return (b,) + _ptr(per)
    return _layout(name)


def _rows(batch, D, dtype, seed):
    """Sentence rows with many exact ties: even columns on a 0.5 grid (zeros included), odd columns continuous."""
    x = torch.randn(batch.n_rows, D, generator=torch.Generator().manual_seed(seed))
    x[:, ::2] = torch.round(x[:, ::2] * 2) / 2
    return x.to(dtype).to(DEV)


def _case(name, D, dtype, seed=1):
    import ed_gated_gcn_b200 as E
    batch, pp, an = _layout_m(name)
    graph = _graph(batch)
    pairs = E.pairs_from_ptr(graph, torch.from_numpy(pp), torch.from_numpy(an))
    eb, rows = _expand(batch, pp, an)
    return batch, graph, pairs, eb, _graph(eb), rows, an, _rows(batch, D, dtype, seed)


def _t_pads(batch, pp, an):
    """The longest sentence with a pair, 3 more, and a value with a + 1 == T_pad for a pair in the middle."""
    owner = np.repeat(np.arange(batch.n_graphs), np.diff(pp))
    T = int(batch.lengths[owner].max())
    return [T, T + 3, int(an[len(an) // 2]) + 1]


def _sentence_arg(arg_e, rows):
    """Expanded-batch arg rows mapped back to sentence rows (-1 stays)."""
    a = arg_e.long().cpu()
    return torch.where(a >= 0, rows[a.clamp_min(0)], torch.full_like(a, -1)).int()


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
@pytest.mark.parametrize("D", [24, 300, 768])
@pytest.mark.parametrize("layout", LAYOUTS)
def test_forward_bit_exact_against_the_expanded_batch(layout, D, dtype):
    import ed_gated_gcn_b200 as E
    batch, graph, pairs, eb, eg, rows, an, h = _case(layout, D, dtype)
    he = h[rows.to(DEV)]
    ea = torch.from_numpy(eb.anchor)
    for T in _t_pads(batch, pairs.pair_ptr.cpu().numpy(), an):
        got, arg = E.lr_pool(h, graph, pairs.anchor, T_pad=T, return_arg=True, pairs=pairs)
        want, arg_e = E.lr_pool(he, eg, ea, T_pad=T, return_arg=True)
        assert got.shape == (len(an), 2 * D) and arg.shape == (len(an), 2 * D)
        assert torch.equal(got, want), T
        assert torch.equal(arg.cpu(), _sentence_arg(arg_e, rows)), T


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
@pytest.mark.parametrize("D", [24, 300, 768])
@pytest.mark.parametrize("layout", LAYOUTS)
def test_gradient_is_the_expanded_gradient_summed_over_pairs(layout, D, dtype):
    import ed_gated_gcn_b200 as E
    batch, graph, pairs, eb, eg, rows, an, h = _case(layout, D, dtype, seed=2)
    T = _t_pads(batch, pairs.pair_ptr.cpu().numpy(), an)[0]
    probe = torch.randn(len(an), 2 * D, generator=torch.Generator().manual_seed(3)).to(DEV)
    hg = h.clone().requires_grad_(True)
    _, arg = E.lr_pool(hg, graph, pairs.anchor, T_pad=T, return_arg=True, pairs=pairs)
    E.lr_pool(hg, graph, pairs.anchor, T_pad=T, pairs=pairs).backward(probe)
    he = h[rows.to(DEV)].clone().requires_grad_(True)
    E.lr_pool(he, eg, torch.from_numpy(eb.anchor), T_pad=T).backward(probe)
    want = torch.zeros(batch.n_rows, D, dtype=torch.float64)
    want.index_add_(0, rows, he.grad.double().cpu())              # fp64, over each sentence's pairs
    got = hg.grad.double().cpu()
    assert hg.grad.dtype == dtype
    if dtype == torch.bfloat16:
        assert rel(got, want) < 1e-2
        return
    assert rel(got, want) < 1e-6
    # contributors per element: exactly one gives the probe value itself, none gives an exact zero
    a = arg.long().cpu()
    col = torch.arange(2 * D).remainder(D).expand_as(a)
    ok = a >= 0
    count = torch.zeros(batch.n_rows * D, dtype=torch.int64)
    count.index_add_(0, (a * D + col)[ok], torch.ones(int(ok.sum()), dtype=torch.int64))
    count = count.view(batch.n_rows, D)
    assert torch.equal(got[count == 1], want[count == 1])
    assert (got[count == 0] == 0).all()


def _crafted():
    """Sentences built to hit every tie rule, with their pairs in no particular order."""
    import ed_gated_gcn_b200 as E
    from ed_gated_gcn_b200 import synth
    D = 24
    g = torch.Generator().manual_seed(4)
    L = [6, 5, 7, 8, 1, 3, 4]
    sents = [torch.randn(n, D, generator=g) for n in L]
    sents[1] = -sents[1].abs() - 0.1                                  # all negative: the masked zeros win
    sents[2][:, :5] = 0.0                                             # exact zeros tying the masked zero
    sents[2][3, 5:9] = 0.0
    sents[3][:, :12] = torch.tensor([1.0, 0.5, 1.0, -2.0, 1.0, 0.25, 1.0, 1.0])[:, None]   # equal maxima: first wins
    sents[6][:, :6] = -1.0
    per = [[5, 0, 2, 0], [4, 0, 2], [3, 6, 0, 3], [1, 4, 7, 4, 0], [0], [], [3, 0]]   # anchors 0 and n - 1 everywhere
    pp, an = _ptr(per)
    batch = synth.make_batch(len(L), 0, 0, seed=5, lengths=np.asarray(L))
    graph = _graph(batch)
    pairs = E.pairs_from_ptr(graph, torch.from_numpy(pp), torch.from_numpy(an))
    return batch, graph, pairs, torch.cat(sents), pp, an, D


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
def test_crafted_ties_against_the_oracle(dtype):
    import ed_gated_gcn_b200 as E
    batch, graph, pairs, x, pp, an, D = _crafted()
    x = x.to(dtype).float()                                           # the oracle sees the values the kernel reads
    owner = np.repeat(np.arange(batch.n_graphs), np.diff(pp))
    sp, lens = batch.sent_ptr, batch.lengths
    T = int(lens.max())
    xd = torch.zeros(len(an), T, D)
    for p, s in enumerate(owner):
        xd[p, :lens[s]] = x[sp[s]:sp[s + 1]]
    anchor, length = torch.from_numpy(an).long(), torch.from_numpy(lens[owner]).long()
    want = O.bertdm_pool_ref(xd, anchor, length)
    h = x.to(dtype).to(DEV).requires_grad_(True)
    got = E.lr_pool(h, graph, pairs.anchor, T_pad=T, pairs=pairs)
    assert torch.equal(got.cpu(), want)
    # gradient routing = torch.max's; an integer probe keeps every sum exact, so the sums compare exactly too
    probe = torch.randint(-4, 5, (len(an), 2 * D), generator=torch.Generator().manual_seed(6)).float()
    xr = xd.clone().requires_grad_(True)
    O.bertdm_pool_ref(xr, anchor, length).backward(probe)
    got.backward(probe.to(DEV))
    want_g = torch.zeros(batch.n_rows, D)
    for p, s in enumerate(owner):
        want_g[sp[s]:sp[s + 1]] += xr.grad[p, :lens[s]]
    assert torch.equal(h.grad.float().cpu(), want_g)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
def test_bertdm_fixture_on_grouped_pairs(dtype):
    """tests/golden/bertdm.npz through wordpiece_mean once per sentence -> lr_pool(pairs=) + trigger rows: the fixture's
    own pair of every sentence reproduces the tensor entering self.dense, with extra pairs per sentence alongside."""
    import ed_gated_gcn_b200 as E
    z = np.load(os.path.join(GOLDEN, "bertdm.npz"))
    lengths, anchor = z["lengths"], z["anchor"]
    B, Lb, D = z["bert_x"].shape
    transform = torch.from_numpy(z["transform"]).to(DEV)
    bert_x = torch.from_numpy(z["bert_x"]).to(DEV).requires_grad_(True)
    s_all, n_all = E.segments_from_transform(transform)
    T = transform.shape[1]
    keep = torch.cat([torch.arange(int(n)) + b * T for b, n in enumerate(lengths)]).to(DEV)
    words = E.wordpiece_mean(bert_x.reshape(B * Lb, D), s_all[keep], n_all[keep], compute_dtype=dtype)
    sent_ptr = torch.from_numpy(np.concatenate([[0], np.cumsum(lengths)]).astype(np.int32))
    heads = torch.cat([torch.cat([torch.tensor([-1]), torch.arange(int(n) - 1)]) for n in lengths])
    graph = E.build_graph(heads, sent_ptr, device=DEV)
    rng = np.random.default_rng(8)
    per, fixture_pair = [], []
    for b, n in enumerate(lengths):
        extra = list(rng.integers(0, int(n), size=3)) + [int(n) - 1, 0]
        fixture_pair.append(sum(len(p) for p in per) + 2)           # the fixture's pair sits among the extra ones
        per.append(extra[:2] + [int(anchor[b])] + extra[2:])
    pp, an = _ptr(per)
    pairs = E.pairs_from_ptr(graph, torch.from_numpy(pp), torch.from_numpy(an))
    pooled = E.lr_pool(words, graph, pairs.anchor, pairs=pairs)      # T_pad = graph.max_len = lengths.max()
    trig = words[(pairs.pair_start + pairs.anchor).long()]           # the trigger row of every pair
    dense_in = torch.cat([trig.float(), pooled], 1)
    fp = torch.tensor(fixture_pair, device=DEV)
    tol = 1e-6 if dtype == torch.float32 else 1e-2
    assert rel(dense_in[fp], z["dense_in"]) < tol
    # the extra pairs equal the per-sentence call on the expanded batch
    owner = np.repeat(np.arange(B), np.diff(pp))
    spn = sent_ptr.numpy()
    rows = torch.from_numpy(np.concatenate([np.arange(spn[s], spn[s + 1]) for s in owner])).to(DEV)
    ep = torch.from_numpy(np.concatenate([[0], np.cumsum(lengths[owner])]).astype(np.int32))
    eg = E.build_graph(torch.cat([heads[sent_ptr[s]:sent_ptr[s + 1]] for s in owner]), ep, device=DEV)
    assert torch.equal(pooled, E.lr_pool(words[rows], eg, torch.from_numpy(an), T_pad=int(lengths.max())))
    # gradient w.r.t. the BERT output: the probe on the fixture's pairs, zero on the others
    g = torch.zeros_like(dense_in)
    g[fp] = torch.from_numpy(z["probe"]).to(DEV)
    dense_in.backward(g)
    if dtype == torch.float32:
        assert rel(bert_x.grad, z["d_bert_x"]) < 1e-6
    else:
        assert rel(bert_x.grad.float().sum(1).cpu(), torch.from_numpy(z["d_bert_x"]).sum(1)) < 2e-2


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
def test_deterministic_and_captured(dtype):
    """Two runs are bitwise equal; a captured forward + backward replays to the eager result."""
    import ed_gated_gcn_b200 as E
    from ed_gated_gcn_b200.runtime import GraphedStep
    batch, graph, pairs, eb, eg, rows, an, h = _case("outside-plan", 300, dtype)
    h = h.requires_grad_(True)
    probe = torch.randn(len(an), 600, generator=torch.Generator().manual_seed(9)).to(DEV)
    res = {}

    def step():
        h.grad = None
        pooled, arg = E.lr_pool(h, graph, pairs.anchor, return_arg=True, pairs=pairs)
        pooled.backward(probe)
        res.update(pooled=pooled.detach(), arg=arg, dh=h.grad)
        return pooled

    step()
    first = {k: v.clone() for k, v in res.items()}
    step()
    for k, v in first.items():
        assert torch.equal(res[k], v), k
    gs = GraphedStep(step)
    for k in res:
        res[k].zero_()
    gs()
    torch.cuda.synchronize()
    for k, v in first.items():
        assert torch.equal(res[k], v), k


def test_edge_and_error_cases():
    import ed_gated_gcn_b200 as E
    batch, pp, an = _layout("mixed")
    graph = _graph(batch)
    D = 24
    h = torch.randn(batch.n_rows, D, device=DEV).requires_grad_(True)
    # no pairs at all: [0, 2D], and a zero gradient on every row
    none = E.pairs_from_ptr(graph, torch.zeros(batch.n_graphs + 1, dtype=torch.int32), torch.zeros(0, dtype=torch.int32))
    out = E.lr_pool(h, graph, none.anchor, pairs=none)
    assert out.shape == (0, 2 * D)
    out.sum().backward()
    assert h.grad is not None and torch.equal(h.grad, torch.zeros_like(h))
    pairs = E.pairs_from_ptr(graph, torch.from_numpy(pp), torch.from_numpy(an))
    with pytest.raises(E.EdgError, match="one anchor per pair"):
        E.lr_pool(h, graph, pairs.anchor[:-1], pairs=pairs)
    other = _graph(_lengths_batch([4, 5], seed=1))
    op = E.pairs_from_ptr(other, torch.tensor([0, 1, 2]), torch.tensor([0, 4]))
    with pytest.raises(E.EdgError, match="sentences"):
        E.lr_pool(h, graph, op.anchor, pairs=op)
    with pytest.raises(E.EdgError, match="every sentence once"):
        E.lr_pool(h[:-1], graph, pairs.anchor, pairs=pairs)
    with pytest.raises(E.EdgError, match="CUDA"):
        E.lr_pool(h.detach().cpu(), graph, pairs.anchor, pairs=pairs)
