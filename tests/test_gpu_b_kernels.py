"""Floating-point kernels one by one, through the C ABI, against CPU torch fp32/fp64.
fp32 mode: <= 1e-5 relative (max|a-b| / max|b|); bf16 mode: <= 2e-2 relative."""
import numpy as np
import pytest
import torch

from gpu_util import DEV, rel, tol_for, dense_inputs, pack_rows
from oracle import ref_oracle as O

pytestmark = pytest.mark.gpu
DTYPES = [torch.float32, torch.bfloat16]


def _batch_graph(B, lo, hi, seed, skewed=False):
    import ed_gated_gcn_b200 as E
    from ed_gated_gcn_b200 import synth
    batch = synth.make_batch(B, lo, hi, seed=seed, skewed=skewed)
    g = E.build_graph(torch.from_numpy(batch.heads), torch.from_numpy(batch.sent_ptr), device=DEV)
    return batch, g


@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "bf16"])
@pytest.mark.parametrize("D", [300, 256, 8, 20])
def test_aggregate_forward_and_transpose(dtype, D):
    from ed_gated_gcn_b200 import ops
    batch, g = _batch_graph(37, 1, 50, seed=D)
    x = torch.randn(batch.n_rows, D)
    xr = ops.as_rows(x.to(DEV), dtype)
    x_used = xr.float().cpu()
    # oracle: per sentence, exact-size adjacency (packed mode has no pad rows)
    want, want_t = [], []
    for b, h in enumerate(batch.heads_list()):
        lo, hi = batch.sent_ptr[b], batch.sent_ptr[b + 1]
        a = torch.from_numpy(O.dense_adjacency_from_heads(h, len(h))).float()
        xs = x_used[lo:hi]
        den = a.sum(1, keepdim=True) + 1
        want.append((a @ xs) / den)                  # gcn.py:35,41
        want_t.append(a.t() @ (xs / den))            # its adjoint
    y = ops.aggregate(xr, g, mode=0)
    yt = ops.aggregate(xr, g, mode=1)
    assert rel(y.float(), torch.cat(want)) < (1e-6 if dtype == torch.float32 else 8e-3)
    assert rel(yt.float(), torch.cat(want_t)) < (1e-6 if dtype == torch.float32 else 8e-3)
    # mixed dtype output path
    y32 = ops.aggregate(xr, g, mode=0, out_dtype=torch.float32)
    assert rel(y32, torch.cat(want)) < 1e-6


@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "bf16"])
@pytest.mark.parametrize("shape", [(1, 16, 16), (127, 300, 300), (128, 64, 256), (1000, 300, 300), (513, 768, 768),
                                   (4096, 256, 256), (77, 40, 24), (300, 304, 8)])
@pytest.mark.parametrize("act", [0, 1])
def test_linear(dtype, shape, act):
    from ed_gated_gcn_b200 import ops
    M, K, Nout = shape
    g = torch.Generator().manual_seed(M + K)
    a = torch.randn(M, K, generator=g)
    w = torch.randn(Nout, K, generator=g) / K ** 0.5
    bias = torch.randn(Nout, generator=g)
    ar, wr = ops.as_rows(a.to(DEV), dtype), ops.as_rows(w.to(DEV), dtype)
    want = ar.float().cpu().double() @ wr.float().cpu().double().t() + bias.double()
    if act == 1:
        want = torch.sigmoid(want)
    for out_dtype in (dtype, torch.float32):
        got = ops.linear(ar, wr, bias.to(DEV), act=act, out_dtype=out_dtype)
        tol = 2e-6 if out_dtype == torch.float32 else 5e-3
        assert rel(got.float(), want) < tol, (shape, out_dtype)
        # the row padding must stay finite/zero: later kernels read whole 16-byte chunks
        base = got.as_strided((M, got.stride(0)), (got.stride(0), 1))
        assert torch.isfinite(base.float()).all()
        assert (base[:, Nout:] == 0).all()


@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "bf16"])
@pytest.mark.parametrize("shape", [(50, 16, 16), (1000, 300, 300), (4096, 256, 256), (3000, 768, 768), (129, 300, 40),
                                   (64, 8, 304), (20000, 300, 300), (16000, 256, 128), (9600, 100, 24), (12000, 384, 160)])
def test_wgrad(dtype, shape):
    from ed_gated_gcn_b200 import ops
    R, K1, K2 = shape
    g = torch.Generator().manual_seed(R + K1)
    a = torch.randn(R, K1, generator=g)
    b = torch.randn(R, K2, generator=g)
    ar, br = ops.as_rows(a.to(DEV), dtype), ops.as_rows(b.to(DEV), dtype)
    ad, bd = ar.float().cpu().double(), br.float().cpu().double()
    for bias_of in (0, 1, 2):
        dW, db = ops.wgrad(ar, br, bias_of=bias_of)
        assert rel(dW, ad.t() @ bd) < 2e-6
        if bias_of == 1:
            assert rel(db, ad.sum(0)) < 2e-6
        if bias_of == 2:
            assert rel(db, bd.sum(0)) < 2e-6


@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "bf16"])
def test_tensor_core_kernels_agree_with_ffma_kernels(dtype, monkeypatch):
    """bf16: tcgen05 results vs torch on the same bf16 inputs at a full-size shape (C2 rows)."""
    if dtype != torch.bfloat16:
        pytest.skip("tensor-core path is bf16 only")
    from ed_gated_gcn_b200 import ops
    M, K, Nout = 112_640, 300, 300
    g = torch.Generator().manual_seed(1)
    a = ops.as_rows(torch.randn(M, K, generator=g).to(DEV), dtype)
    w = ops.as_rows((torch.randn(Nout, K, generator=g) / K ** 0.5).to(DEV), dtype)
    got = ops.linear(a, w, None, out_dtype=torch.float32)
    want = a.float() @ w.float().t()                   # cuBLAS fp32 as the on-device checker
    assert rel(got, want) < 1e-5
    dW, _ = ops.wgrad(a, a)
    assert rel(dW, a.float().t() @ a.float()) < 2e-5


@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "bf16"])
def test_pool_views_ties_and_diversity(dtype):
    from ed_gated_gcn_b200 import ops
    batch, g = _batch_graph(21, 1, 30, seed=4)
    D, V = 40, 3
    h = torch.randn(batch.n_rows, D)
    h[batch.sent_ptr[3]:batch.sent_ptr[4]] = 0.25              # a sentence of identical rows: first row must win
    gates = torch.rand(V, batch.n_graphs, D) + 0.05
    hr = ops.as_rows(h.to(DEV), dtype)
    pooled, arg = ops.pool_fwd(hr, g, gates.to(DEV))
    hu = hr.float().cpu()
    for b in range(batch.n_graphs):
        lo, hi = int(batch.sent_ptr[b]), int(batch.sent_ptr[b + 1])
        for v in range(V):
            val, idx = torch.max(hu[lo:hi] * gates[v, b][None, :], dim=0)
            assert torch.equal(pooled[v, b].cpu(), val)
            if b == 3:
                assert (arg[v, b].cpu() == lo).all()
            else:
                assert torch.equal(arg[v, b].cpu().long(), idx + lo)
    xy = ops.diversity_fwd(pooled)
    p = pooled.double().cpu()
    want = sum((p[i] * p[j]).sum(1).mean() for i in range(V) for j in range(i + 1, V))
    assert rel(xy, want) < 1e-6


@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "bf16"])
@pytest.mark.parametrize("i64", [False, True])
def test_scores_kl(dtype, i64):
    from ed_gated_gcn_b200 import ops
    import ed_gated_gcn_b200 as E
    batch, g = _batch_graph(19, 1, 45, seed=8)
    D = 300
    B = batch.n_graphs
    h = ops.as_rows(torch.randn(batch.n_rows, D).to(DEV), dtype)
    gate = torch.rand(B, D); v = torch.randn(B, D) * 0.1; c = torch.randn(B)
    dist = E.tree_distance(g, torch.from_numpy(batch.anchor).to(DEV))
    if i64:
        dist = dist.long()
    scores, kl_b, kl = ops.scores_kl_fwd(h, g, gate.to(DEV), v.to(DEV), c.to(DEV), dist)
    hu = h.float().cpu().double()
    for b in range(B):
        lo, hi = int(batch.sent_ptr[b]), int(batch.sent_ptr[b + 1])
        s = (hu[lo:hi] * gate[b].double() * v[b].double()).sum(1) + c[b].double()
        assert rel(scores[lo:hi], s) < 2e-6
        q = torch.softmax(dist[lo:hi].cpu().double(), 0)
        want = (torch.softmax(s, 0) * q).sum()
        assert abs(kl_b[b].item() - want.item()) < 2e-6
    assert abs(kl.item() - kl_b.double().mean().item()) < 1e-6


@pytest.mark.parametrize("shape", [(4096, 300, 34), (37, 256, 2), (1, 16, 1), (130, 768, 34), (64, 300, 64)])
def test_block_head_fc_only_forward_backward(shape):
    """[v | va] = logits @ fc.weight, c = a.va + logits.fc.bias (bert_amir5.py:645-646 collapsed) and its
    backward, against the torch formulation in fp64: the block head's launches without the dense head (the logits of
    a torch logits_fn as input), the parameter gradients from edg_block_head_wgrad without d logits."""
    from ed_gated_gcn_b200 import ops
    B, D, C = shape
    g = torch.Generator().manual_seed(B + D + C)
    lg, W, bfc = torch.randn(B, C, generator=g), torch.randn(C, 2 * D, generator=g) / C ** 0.5, torch.randn(C, generator=g)
    a, dv, dc = torch.randn(B, D, generator=g), torch.randn(B, D, generator=g), torch.randn(B, generator=g)
    lg_, W_, bfc_, a_, dv_, dc_ = (t.to(DEV) for t in (lg, W, bfc, a, dv, dc))
    _, lg_out, v, c = ops.block_head_fwd(a_, a_, None, None, None, None, W_, bfc_, logits=lg_)
    assert torch.equal(lg_out, lg_)
    lgd, Wd, bd, ad = (t.double().requires_grad_(True) for t in (lg, W, bfc, a))
    vva = lgd @ Wd
    v_ref = vva[:, :D]
    c_ref = (ad * vva[:, D:]).sum(1) + lgd @ bd
    assert rel(v, v_ref) < 1e-6 and rel(c, c_ref) < 1e-6
    for scale in (None, 0.37):
        s = 1.0 if scale is None else scale
        want = torch.autograd.grad([v_ref, c_ref], [lgd, ad, Wd, bd], [s * dv.double(), s * dc.double()], retain_graph=True)
        sc = None if scale is None else torch.tensor(scale, device=DEV)
        d_lg, d_a, dp = ops.block_head_bwd(lg_, a_, a_, False, None, W_, bfc_, dv_, dc_, sc)
        _, _, d_fw, d_fb = ops.block_head_wgrad(lg_, None, a_, a_, None, dv_, dc_, sc)
        assert dp is None
        for name, x, y in zip(["d_logits", "d_a", "d_fc_w", "d_fc_b"], (d_lg, d_a, d_fw, d_fb), want):
            assert rel(x, y) < 2e-6, (name, shape, scale)
        # where the modes overlap (a dense head of zeros adds exact zeros to d a), the combined launches give the
        # same bits
        zw, p = torch.zeros_like(W_), torch.randn(B, D, generator=g).to(DEV)
        dlg2, da2, _ = ops.block_head_bwd(lg_, a_, a_, False, zw, W_, bfc_, dv_, dc_, sc)
        _, _, d_fw2, d_fb2 = ops.block_head_wgrad(lg_, dlg2, a_, a_, p, dv_, dc_, sc)
        assert torch.equal(dlg2, d_lg) and torch.equal(da2, d_a)
        assert torch.equal(d_fw2, d_fw) and torch.equal(d_fb2, d_fb)


@pytest.mark.parametrize("D", [300, 256, 200, 64, 320])
@pytest.mark.parametrize("B", [4096, 77])
@pytest.mark.parametrize("pairs", [2, 3])
def test_mlp_chain_forward_backward(D, B, pairs):
    """The fused gate-MLP launch against torch on the same bf16-rounded operands (fp32 accumulation)."""
    from ed_gated_gcn_b200 import ops
    bf = torch.bfloat16
    G = 2
    g = torch.Generator().manual_seed(D + B + pairs)
    s0 = ops.as_rows(torch.rand(B, D, generator=g).to(DEV), bf)
    Ws = [[ops.as_rows((torch.randn(D, D, generator=g) * 2 / D ** 0.5).to(DEV), bf) for _ in range(pairs)] for _ in range(G)]
    bs = [[torch.randn(D, generator=g).to(DEV) for _ in range(pairs)] for _ in range(G)]
    gates = torch.empty(G, B, D, device=DEV)
    acts = [[s0] for _ in range(G)]
    stages = []
    for k in range(G):
        st = []
        for i in range(pairs):
            last = i == pairs - 1
            out = gates[k] if last else ops.alloc_rows(B, D, bf, DEV)
            st.append(dict(w=Ws[k][i], bias=bs[k][i], out=out))
            if not last:
                acts[k].append(out)
        stages.append(st)
    ops.mlp_chain(0, [s0] * G, stages, B, D)
    for k in range(G):
        s = s0.float()
        for i in range(pairs):
            s = torch.sigmoid(s @ Ws[k][i].float().t() + bs[k][i])
            if i < pairs - 1:
                got = acts[k][i + 1]
                assert rel(got.float(), s) < 6e-3, ("act", D, B, k, i)
                base = got.as_strided((B, got.stride(0)), (got.stride(0), 1))
                assert (base[:, D:] == 0).all()                      # padding columns stay zero
                s = got.float()                                       # the kernel feeds the rounded tile forward
        assert rel(gates[k], s) < 2e-5, ("gate", D, B, k)
    # backward chain: dz_last -> ... -> d a, with sigmoid' of the saved activations
    dz = [ops.as_rows(torch.randn(B, D, generator=g).to(DEV), bf) for _ in range(G)]
    Wt = [[ops.as_rows(Ws[k][i].float().t().contiguous(), bf) for i in range(pairs)] for k in range(G)]
    da = torch.empty(G, B, D, device=DEV)
    mids = [[None] * pairs for _ in range(G)]
    stages = []
    for k in range(G):
        st = []
        for i in range(pairs - 1, -1, -1):
            if i > 0:
                out = ops.alloc_rows(B, D, bf, DEV)
                mids[k][i - 1] = out
                st.append(dict(w=Wt[k][i], y=acts[k][i], out=out))
            else:
                st.append(dict(w=Wt[k][0], y=acts[k][0] if k == 0 else None, out=da[k]))
        stages.append(st)
    ops.mlp_chain(1, dz, stages, B, D)
    for k in range(G):
        d = dz[k].float()
        for i in range(pairs - 1, -1, -1):
            ds = d @ Wt[k][i].float().t()
            if i > 0:
                y = acts[k][i].float()
                want = ds * y * (1 - y)
                assert rel(mids[k][i - 1].float(), want) < 6e-3, ("dz", D, B, k, i)
                d = mids[k][i - 1].float()
            else:
                y = acts[k][0].float()
                want = ds * y * (1 - y) if k == 0 else ds
                assert rel(da[k], want) < 2e-5, ("da", D, B, k)


@pytest.mark.parametrize("shape", [(4096, 300, 300, 4), (130, 256, 256, 2), (1000, 64, 200, 8), (4096, 300, 300, 1)])
def test_wgrad_batch(shape):
    from ed_gated_gcn_b200 import ops
    R, K1, K2, n = shape
    g = torch.Generator().manual_seed(R + n)
    a = [ops.as_rows(torch.randn(R, K1, generator=g).to(DEV), torch.bfloat16) for _ in range(n)]
    b = [ops.as_rows(torch.randn(R, K2, generator=g).to(DEV), torch.bfloat16) for _ in range(n)]
    for bias_of in (0, 1, 2):
        dWs, dbs = ops.wgrad_batch(a, b, bias_of=bias_of)
        for i in range(n):
            ad, bd = a[i].float().double(), b[i].float().double()
            assert rel(dWs[i], ad.t() @ bd) < 2e-6
            if bias_of == 1:
                assert rel(dbs[i], ad.sum(0)) < 2e-6
            if bias_of == 2:
                assert rel(dbs[i], bd.sum(0)) < 2e-6


@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "bf16"])
@pytest.mark.parametrize("long_sentences", [False, True])
def test_pool_fwd_hmax_is_the_column_maximum(dtype, long_sentences):
    """edg_pool_fwd's optional hmax is the plain column maximum of every sentence, whatever the gates (one exactly 0)."""
    from ed_gated_gcn_b200 import ops
    batch, g = _batch_graph(6 if long_sentences else 45, 300 if long_sentences else 1, 700 if long_sentences else 40, seed=17)
    D, V, B = 76, 2, batch.n_graphs
    gen = torch.Generator().manual_seed(3)
    h = ops.as_rows(torch.randn(batch.n_rows, D, generator=gen).to(DEV), dtype)
    gates = (torch.rand(V, B, D, generator=gen) + 0.05).to(DEV)
    gates[1, 2, :7] = 0.0                                       # an exactly-zero gate
    _, _, hmax = ops.pool_fwd(h, g, gates, want_hmax=True)
    hu = h.float()
    for b in (0, 2, B - 1):
        lo, hi = int(batch.sent_ptr[b]), int(batch.sent_ptr[b + 1])
        assert torch.equal(hmax[b], hu[lo:hi].max(0)[0])


@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "bf16"])
def test_views_bwd_in_halves_equals_one_call(dtype):
    """edg_views_bwd_parts: the dh half and the dgates half issued separately give the bits of the single call."""
    from ed_gated_gcn_b200 import ops
    batch, g = _batch_graph(30, 1, 35, seed=23)
    D, V, B = 48, 3, batch.n_graphs
    gen = torch.Generator().manual_seed(5)
    h = ops.as_rows(torch.randn(batch.n_rows, D, generator=gen).to(DEV), dtype)
    gates = (torch.rand(V, B, D, generator=gen) + 0.05).to(DEV)
    pooled, arg = ops.pool_fwd(h, g, gates)
    g_xy = torch.tensor(1.3, device=DEV)
    dh0 = ops.as_rows(torch.randn(batch.n_rows, D, generator=gen).to(DEV), dtype)
    base = torch.randn(V, B, D, generator=gen).to(DEV)
    dh_a, dg_a = dh0.clone(), base.clone()
    ops.views_bwd(pooled, arg, gates, h, g_xy, None, dh_a, dg_a, acc_view=2)
    dh_b, dg_b = dh0.clone(), base.clone()
    ops.views_bwd(pooled, arg, gates, h, g_xy, None, None, dg_b, acc_view=2, parts=2)
    ops.views_bwd(pooled, arg, gates, h, g_xy, None, dh_b, None, parts=1)
    assert torch.equal(dh_a, dh_b) and torch.equal(dg_a, dg_b)
    assert not torch.equal(dh_a, dh0)


def test_fused_adam_matches_torch_adam():
    """edg_adam_multi (one launch for all tensors, device step counter) against torch.optim.Adam, the optimiser of
    train.py:239-243, over several steps incl. tensors that are not a multiple of the 1024-element chunk."""
    import ed_gated_gcn_b200 as E
    gen = torch.Generator().manual_seed(5)
    shapes = [(300, 300), (300,), (34, 600), (1,), (1025,), (7, 3)] + [(17,)] * 30       # > 32 tensors: two launches
    ref = [torch.nn.Parameter(torch.randn(*s, generator=gen).to(DEV)) for s in shapes]
    mine = [torch.nn.Parameter(p.detach().clone()) for p in ref]
    o_ref = torch.optim.Adam(ref, lr=1e-2, betas=(0.9, 0.999), eps=1e-8)
    o_mine = E.FusedAdam(mine, lr=1e-2, betas=(0.9, 0.999), eps=1e-8)
    for step in range(5):
        for a, b in zip(ref, mine):
            g = torch.randn(a.shape, generator=gen).to(DEV) * (10.0 ** (step - 2))
            a.grad, b.grad = g.clone(), g.clone()
        if step == 3:
            ref[1].grad = None; mine[1].grad = None            # a parameter without gradient is skipped
        o_ref.step(); o_mine.step()
        for a, b in zip(ref, mine):
            assert rel(b, a) < 2e-6, (step, tuple(a.shape))
    assert o_mine.step_count.tolist() == [5.0, 4.0] + [5.0] * (len(shapes) - 2)
    with pytest.raises(E.EdgError):
        E.FusedAdam([torch.nn.Parameter(torch.zeros(3))])      # CPU parameter: no fallback


# ---------------------------------------------------------------------------------------------
# fp32-parity GEMMs on the tensor cores: split operands (csrc/edg_split.cu, include/edgcn.h)
# ---------------------------------------------------------------------------------------------
def _wide_rows(M, K, seed, scale=1.0):
    """fp32 rows whose magnitudes span several orders (per-row factors e^N(0,2)): what a per-tensor scale must survive"""
    g = torch.Generator().manual_seed(seed)
    return torch.randn(M, K, generator=g) * torch.exp(2 * torch.randn(M, 1, generator=g)) * scale


@pytest.mark.parametrize("shape", [(1, 8), (1000, 300), (777, 64), (300, 65), (0, 300)])
@pytest.mark.parametrize("scale", [1.0, 1e-20, 3e18])
def test_split_rows_reconstruct_the_fp32_matrix(shape, scale):
    from ed_gated_gcn_b200 import ops
    M, K = shape
    x = _wide_rows(M, K, seed=M + K, scale=scale)
    s = ops.split_rows(x.to(DEV))
    kp = s.data.shape[1] // 2
    assert kp % 64 == 0 and kp >= K and s.shape == (M, K)
    if M == 0:
        assert float(s.amax) == 0.0
        return
    amax = float(s.amax)
    assert amax == float(x.abs().max())
    e = int(np.floor(np.log2(amax))) + 1                      # amax in [2^(e-1), 2^e)
    sc = 2.0 ** (14 - e)
    d = s.data[:M].double().cpu()
    hi, lo = d[:, :kp], d[:, kp:]
    assert (hi[:, K:] == 0).all() and (lo[:, K:] == 0).all()  # the padding the TMA boxes read
    assert hi.abs().max() < 2 ** 14
    back = (hi[:, :K] + lo[:, :K]) / sc
    err = (back - x.double()).abs()
    # 22 significant bits, absolute floor 2^-25 in scaled units
    assert bool((err <= torch.maximum(x.double().abs() * 2.0 ** -21, torch.tensor(2.0 ** -24 / sc, dtype=torch.float64))).all())


@pytest.mark.parametrize("shape", [(4096, 300, 300), (1025, 64, 48), (1500, 130, 520), (5000, 300, 20), (2047, 768, 768),
                                   (112_640, 300, 300)])
@pytest.mark.parametrize("act", [0, 2])
def test_linear_split_matches_fp64(shape, act):
    from ed_gated_gcn_b200 import ops
    M, K, Nout = shape
    a = _wide_rows(M, K, seed=M)
    g = torch.Generator().manual_seed(K)
    w = torch.randn(Nout, K, generator=g) / K ** 0.5
    bias = torch.randn(Nout, generator=g)
    assert ops.f32_tc(M, K, Nout)
    ad = a.to(DEV)
    got = ops.linear_split(ops.split_rows(ad), ops.split_rows(w.to(DEV)), bias.to(DEV), act=act)
    want = ad.double() @ w.to(DEV).double().t() + bias.to(DEV).double()
    if act == 2:
        want = want.clamp_min(0)
    assert rel(got, want) < 3e-6, shape          # fp32 accumulation in TMEM truncates: ~1e-6 at K = 300
    # row by row: a row 1e4 times smaller than the largest one still has to be right on its own scale
    row_err = (got.double() - want).abs().amax(1) / want.abs().amax(1).clamp_min(1e-30)
    assert float(row_err.max()) < 1e-4
    base = got.as_strided((M, got.stride(0)), (got.stride(0), 1))
    assert (base[:, Nout:] == 0).all()
    # ops.linear takes the same route for fp32 operands of this size
    assert torch.equal(ops.linear(ad, w.to(DEV), bias.to(DEV), act=act), got)


@pytest.mark.parametrize("shape", [(4096, 256, 256), (3000, 768, 768), (20000, 300, 300), (1100, 300, 40), (9600, 100, 24),
                                   (204_800, 300, 300)])
def test_wgrad_split_matches_fp64(shape):
    from ed_gated_gcn_b200 import ops
    R, K1, K2 = shape
    a = _wide_rows(R, K1, seed=R).to(DEV)
    b = _wide_rows(R, K2, seed=R + 1, scale=1e-6).to(DEV)
    a2, b2 = ops.split_rows(a), ops.split_rows(b)
    ad, bd = a.double(), b.double()
    want = ad.t() @ bd
    for bias_of in (0, 1, 2):
        dW, db = ops.wgrad_split(a2, b2, bias_of=bias_of)
        assert rel(dW, want) < 5e-6, (shape, bias_of)
        if bias_of == 1:
            assert rel(db, ad.sum(0)) < 2e-6
        if bias_of == 2:
            assert rel(db, bd.sum(0)) < 2e-6


def test_fp32_ffma_kernels_still_cover_the_large_shapes(monkeypatch):
    """EDG_F32_TC=0 (and every shape the split kernels do not take) keeps the FFMA kernels"""
    from ed_gated_gcn_b200 import ops
    monkeypatch.setenv("EDG_F32_TC", "0")
    assert not ops.f32_tc(4096, 300, 300)
    g = torch.Generator().manual_seed(5)
    a, w = torch.randn(4096, 300, generator=g).to(DEV), (torch.randn(300, 300, generator=g) / 17).to(DEV)
    assert rel(ops.linear(a, w, None), a.double() @ w.double().t()) < 2e-6
    dW, db = ops.wgrad(a, a, bias_of=2)
    assert rel(dW, a.double().t() @ a.double()) < 2e-6 and rel(db, a.double().sum(0)) < 2e-6


# ---------------------------------------------------------------------------------------------
# classifier head + loss (csrc/edg_dense_head.cu): bert_amir5.py:643 self.dense, train.py:121 criterion
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape", [(4096, 300, 34), (33, 300, 34), (1, 64, 2), (257, 768, 34), (100, 20, 7), (64, 300, 50)])
def test_dense_head_forward_backward_vs_torch(shape):
    import ed_gated_gcn_b200 as E
    B, D, C = shape
    g = torch.Generator().manual_seed(B + D)
    a = torch.randn(B, D, generator=g).to(DEV).requires_grad_(True)
    p = torch.randn(B, D, generator=g).to(DEV).requires_grad_(True)
    head = E.DenseHead(2 * D, C).to(DEV)
    probe = torch.randn(B, C, generator=g).to(DEV)
    got = head(a, p)
    (got * probe).sum().backward()
    mine = [a.grad.clone(), p.grad.clone(), head.weight.grad.clone(), head.bias.grad.clone()]
    a.grad = p.grad = None
    head.zero_grad()
    ad, pd_ = a.detach().double().requires_grad_(True), p.detach().double().requires_grad_(True)
    wd, bd = head.weight.detach().double().requires_grad_(True), head.bias.detach().double().requires_grad_(True)
    want = torch.cat([ad, pd_], 1) @ wd.t() + bd                        # the reference's self.dense(cat[...])
    (want * probe.double()).sum().backward()
    assert rel(got, want) < 2e-6
    for m, w in zip(mine, [ad.grad, pd_.grad, wd.grad, bd.grad]):
        assert rel(m, w) < 2e-6
    # plain nn.Linear call (one concatenated argument) still works, same numbers
    assert rel(head(torch.cat([a, p], 1)), want) < 2e-6


@pytest.mark.parametrize("B,C", [(4096, 34), (7, 3), (1, 2), (5000, 64), (300, 1000)])
def test_cross_entropy_matches_torch(B, C):
    import ed_gated_gcn_b200 as E
    g = torch.Generator().manual_seed(B + C)
    logits = (4 * torch.randn(B, C, generator=g)).to(DEV).requires_grad_(True)
    tgt = torch.randint(0, C, (B,), generator=g).to(DEV)
    if B > 4:
        tgt[1::5] = -100                                               # nn.CrossEntropyLoss's ignore_index
    w = torch.tensor(0.37, device=DEV)
    loss = E.cross_entropy(logits, tgt)
    (loss * w).backward()
    got_g = logits.grad.clone()
    logits.grad = None
    ref = torch.nn.functional.cross_entropy(logits.double(), tgt)
    (ref * w.double()).backward()
    assert abs(float(loss) - float(ref)) <= 2e-6 * max(1.0, abs(float(ref)))
    assert rel(got_g, logits.grad) < 5e-6
    assert float(E.CrossEntropyLoss()(logits.detach(), tgt)) == float(loss)
    # every target ignored: zero loss, zero gradient (torch returns nan here; the reference never feeds such a batch)
    logits.grad = None
    l0 = E.cross_entropy(logits, torch.full_like(tgt, -100))
    l0.backward()
    assert float(l0) == 0.0 and float(logits.grad.abs().max()) == 0.0


def test_total_loss_matches_the_torch_expression():
    """train.py:115-118: loss = CE + gate_weight * xy + kl_weight * kl, forward and backward, incl. the ungated xy = 0.0"""
    import ed_gated_gcn_b200 as E
    ce = torch.tensor(1.7, device=DEV, requires_grad=True)
    xy = torch.tensor(0.31, device=DEV, requires_grad=True)
    kl = torch.tensor(2.9, device=DEV, requires_grad=True)
    up = torch.tensor(0.5, device=DEV)
    loss = E.total_loss(ce, xy, kl, 0.01, 0.02)
    (loss * up).backward()
    want = 1.7 + 0.01 * 0.31 + 0.02 * 2.9
    assert abs(float(loss) - want) < 1e-6
    assert abs(float(ce.grad) - 0.5) < 1e-7 and abs(float(xy.grad) - 0.005) < 1e-8 and abs(float(kl.grad) - 0.01) < 1e-8
    ce.grad = None
    loss = E.total_loss(ce, 0.0, kl, 0.01, 0.02)            # BertAmir55NoGate returns xy = 0.0 (a Python float)
    loss.backward()
    assert abs(float(loss) - (1.7 + 0.02 * 2.9)) < 1e-6 and float(ce.grad) == 1.0
