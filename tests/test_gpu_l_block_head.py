"""edg_block_head_fwd / _bwd / _wgrad (the block's classifier head and collapsed-scores algebra, one launch each way)
against fp64 torch, and the combined launches against their dense-only and fc-only modes composed."""
import pytest
import torch

from gpu_util import DEV, rel

pytestmark = pytest.mark.gpu

TOL = 1e-5

# (B, D, C): the flagship shape, then the edges of the tiling -- a partial last block, D = 302 (no 128-bit path),
# D = 768 (several column chunks / passes), C = 2 and C = 64 (the smallest and largest class paddings)
SHAPES = [(4096, 300, 34), (1, 300, 34), (33, 300, 34), (4095, 300, 34), (33, 302, 34), (33, 768, 34), (33, 300, 2),
          (33, 300, 64), (100, 302, 64)]


def _inputs(B, D, C, seed, fc_sigmoid=False):
    g = torch.Generator().manual_seed(seed)
    r = lambda *s: torch.randn(*s, generator=g).to(DEV)
    a = r(B, D)
    t = dict(a=a, af=torch.sigmoid(a) if fc_sigmoid else a, hmax=r(B, D), gate=torch.rand(B, D, generator=g).to(DEV),
             W=r(C, 2 * D) * 0.05, bias=r(C), Wf=r(C, 2 * D) * 0.05, bf=r(C), dv=r(B, D), dc=r(B),
             scale=torch.full((1,), 0.37, device=DEV), g_lg=r(B, C), g_p=r(B, D))
    return t


def _ref(t, fc_sigmoid, scores=True, g_lg=True, g_p=True):
    d = {k: v.double() for k, v in t.items()}
    D = d["a"].shape[1]
    pooled = d["gate"] * d["hmax"]
    lg = torch.cat([d["a"], pooled], 1) @ d["W"].T + d["bias"]
    r = d["af"] @ d["Wf"][:, D:].T
    out = dict(pooled=pooled, logits=lg, v=lg @ d["Wf"][:, :D], c=(lg * (r + d["bf"])).sum(1))
    s = d["scale"][0]
    sdc = s * d["dc"] if scores else torch.zeros_like(d["dc"])
    dlg = d["g_lg"].clone() if g_lg else torch.zeros_like(lg)
    if scores:
        dlg = dlg + (s * d["dv"]) @ d["Wf"][:, :D].T + sdc[:, None] * (r + d["bf"])
    t1 = sdc[:, None] * (lg @ d["Wf"][:, D:])
    if fc_sigmoid:
        t1 = t1 * d["af"] * (1 - d["af"])
    out.update(dlg=dlg, da=t1 + dlg @ d["W"][:, :D], dp=dlg @ d["W"][:, D:] + (d["g_p"] if g_p else 0.0),
               dW=dlg.T @ torch.cat([d["a"], pooled], 1), dbias=dlg.sum(0))
    if scores:
        out.update(dWf=lg.T @ torch.cat([s * d["dv"], sdc[:, None] * d["af"]], 1), dbf=lg.T @ sdc)
    return out


def _run(t, fc_sigmoid, scores=True, g_lg=True, g_p=True):
    from ed_gated_gcn_b200 import ops
    pooled, lg, v, c = ops.block_head_fwd(t["a"], t["af"], t["hmax"], t["gate"], t["W"], t["bias"], t["Wf"], t["bf"])
    sv = (t["dv"], t["dc"], t["scale"]) if scores else (None, None, None)
    dlg, da, dp = ops.block_head_bwd(lg, t["a"], t["af"], fc_sigmoid, t["W"], t["Wf"], t["bf"], *sv,
                                     g_logits=t["g_lg"] if g_lg else None, g_pooled=t["g_p"] if g_p else None)
    dW, dbias, dWf, dbf = ops.block_head_wgrad(lg, dlg, t["a"], t["af"], pooled, *sv)
    return dict(pooled=pooled, logits=lg, v=v, c=c, dlg=dlg, da=da, dp=dp, dW=dW, dbias=dbias, dWf=dWf, dbf=dbf)


@pytest.mark.parametrize("B,D,C", SHAPES)
def test_block_head_equals_fp64(B, D, C):
    t = _inputs(B, D, C, seed=B + D + C)
    got, want = _run(t, False), _ref(t, False)
    for k, w in want.items():
        assert rel(got[k], w) <= TOL, (k, rel(got[k], w))


@pytest.mark.parametrize("B,D,C", [(4096, 300, 34), (33, 302, 34), (33, 768, 64)])
@pytest.mark.parametrize("case", ["fc_sigmoid", "no_scores", "no_g_logits", "no_g_pooled", "only_g_logits"])
def test_block_head_optional_inputs(B, D, C, case):
    fc_sig = case == "fc_sigmoid"
    kw = dict(scores=case not in ("no_scores", "only_g_logits"), g_lg=case != "no_g_logits",
              g_p=case not in ("no_g_pooled", "only_g_logits"))
    t = _inputs(B, D, C, seed=7, fc_sigmoid=fc_sig)
    got, want = _run(t, fc_sig, **kw), _ref(t, fc_sig, **kw)
    for k, w in want.items():
        assert rel(got[k], w) <= TOL, (k, rel(got[k], w))
    if not kw["scores"]:
        assert got["dWf"] is None and got["dbf"] is None


def test_block_head_without_gate_reads_pooled():
    """gate None: pooled is an input (the unfused and the pairs paths pool before the head)."""
    from ed_gated_gcn_b200 import ops
    t = _inputs(33, 300, 34, seed=3)
    pooled = t["gate"] * t["hmax"]
    p2, lg, v, c = ops.block_head_fwd(t["a"], t["af"], pooled, None, t["W"], None, t["Wf"], t["bf"])
    want = _ref(t, False)
    assert p2.data_ptr() == pooled.data_ptr()
    assert rel(lg, want["logits"] - t["bias"].double()) <= TOL
    dW, dbias, _, _ = ops.block_head_wgrad(lg, t["g_lg"], t["a"], t["af"], pooled, want_bias=False)
    assert dbias is None and rel(dW, t["g_lg"].double().T @ torch.cat([t["a"], pooled], 1).double()) <= TOL


@pytest.mark.parametrize("B,D,C", [(4096, 300, 34), (33, 768, 34), (33, 302, 64)])
@pytest.mark.parametrize("fc_sigmoid", [False, True])
def test_block_head_equals_its_two_modes_composed(B, D, C, fc_sigmoid):
    """The same bits as the dense-only and the fc-only launches composed (dense forward -> fc forward on its logits,
    fc backward -> dense backward on its d logits, d a summed, one parameter-gradient launch per head): every sum
    keeps its order in every mode, so a torch head (fc-only) and a DenseHead (combined) give the same training run."""
    from ed_gated_gcn_b200 import ops
    t = _inputs(B, D, C, seed=11, fc_sigmoid=fc_sigmoid)
    got = _run(t, fc_sigmoid)
    sv = (t["dv"], t["dc"], t["scale"])
    pooled, lg, v0, c0 = ops.block_head_fwd(t["a"], None, t["hmax"], t["gate"], t["W"], t["bias"], None, None)
    _, _, v, c = ops.block_head_fwd(t["a"], t["af"], None, None, None, None, t["Wf"], t["bf"], logits=lg)
    dlg, da_fc, dp_fc = ops.block_head_bwd(lg, t["a"], t["af"], fc_sigmoid, None, t["Wf"], t["bf"], *sv,
                                           g_logits=t["g_lg"])
    dlg_d, da_dense, dp = ops.block_head_bwd(None, t["a"], None, False, t["W"], None, None, g_logits=dlg,
                                             g_pooled=t["g_p"])
    dW, dbias, _, _ = ops.block_head_wgrad(None, dlg, t["a"], None, pooled)
    _, _, dWf, dbf = ops.block_head_wgrad(lg, None, t["a"], t["af"], None, *sv)
    assert v0 is None and c0 is None and dp_fc is None and torch.equal(dlg_d, dlg)
    composed = dict(pooled=pooled, logits=lg, v=v, c=c, dlg=dlg, da=da_dense + da_fc, dp=dp, dW=dW, dbias=dbias,
                    dWf=dWf, dbf=dbf)
    for k, w in composed.items():
        assert torch.equal(got[k], w), (k, rel(got[k], w))


@pytest.mark.parametrize("B,D,C", [(4096, 300, 34), (33, 302, 34)])
def test_block_head_is_bitwise_repeatable(B, D, C):
    t = _inputs(B, D, C, seed=5)
    r1, r2 = _run(t, False), _run(t, False)
    for k in r1:
        assert torch.equal(r1[k], r2[k]), k
