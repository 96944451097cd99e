"""The projection and weight-gradient GEMMs at their tile and schedule limits, one kernel at a time, against fp64
references of the stored operands with element-wise bounds.

Kernels and the host rules that pick them (restated below and checked on the CPU):
  bf16 edg_linear   linear_ws (weight tile resident, M >= 512 and the tile fits) or linear_tc (persistent, two TMEM
                    accumulator stages); N tile pick_block_n(Nout, 16), which is an odd multiple of 16 for 368 of the
                    widths 1..1024 (a tile that ends inside its last 32-column epilogue chunk)
  fp32 linear       linear_simt, linear_big (big_linear_ok) or, from F32_TC_MIN_ROWS rows, the split tensor-core path
  edg_wgrad         bf16: wgrad_tc or wgrad_tall (plan_wgrad_tall); fp32: wgrad_simt / wgrad_big (big_wgrad_ok) +
                    split reduce + edg_colsum; edg_wgrad_split: three split launches, the hi x hi one in waves of
                    kSplitMainRows rows
  edg_wgrad_batch, edg_mlp_chain, edg_cast_2d / edg_cast_batch, edg_colsum

Harness, for every case:
  * each output is a view into a NaN-filled allocation with NaN before its first row and at least one guard row
    after its last; after the call the columns < Nout are checked against the reference, the row padding
    [Nout, row_pitch) must be exactly 0 (the padding contract of ops.py) and everything else must still be NaN, so a
    tile that is never written or a store past its tile fails;
  * inputs are column slices of wider allocations whose extra columns hold NaN: the TMA maps take the true K and the
    FFMA loaders bound K, so those columns must never be read;
  * the rows of A and of W carry power-of-two scales in 2^-8 .. 2^8, so a swapped, skipped or duplicated row,
    column or k block lands outside its element's bound;
  * the bound of every element is |got - ref| <= kappa * sum_k |a_k w_k| + rounding of the epilogue, with no
    normalisation by the tensor maximum (see `kappa_*` for the models).

References are fp64 products of the stored operands, formed on the device.
"""
import ctypes

import pytest
import torch

from gpu_util import DEV

NAN = float("nan")
U = 2.0 ** -24                  # unit roundoff of fp32
U_BF16 = 2.0 ** -8              # unit roundoff of bf16
TC_STEP = 2.0 ** -22            # one 16-wide k step of tcgen05 (see kappa_tc)
ACT_ERR = 2.0 ** -21            # __expf / __fdividef in the sigmoid epilogues, absolute
KAPPA_MAX = 2.0 ** -14          # dropping one 16-wide k step must still fail every model below
NUM_SMS = 148
LEAD = 64                       # NaN elements before an output's first row (keeps 16-byte alignment)
ERR = {"OK": 0, "ARG": -1, "DTYPE": -3, "UNSUPPORTED": -7}
TORCH_DT = {"f32": torch.float32, "bf16": torch.bfloat16}
WORST = {}                      # kernel family -> worst |err| / bound seen (printed at the end of the module)


def cdiv(a, b):
    return -(-a // b)


# ------------------------------------------------------------------------------------------------ error models
def kappa_tc(chain):
    """tcgen05 with fp32 accumulation in TMEM: every 16-wide k step adds the aligned sum of 16 exact bf16 / fp16
    products to the accumulator and truncates, once when the products are summed and once when they are added, each
    below 2^-23 of the magnitude reached, which sum_k |a_k w_k| bounds.  `chain` = k elements of the longest chain."""
    k = (cdiv(chain, 16) + 1) * TC_STEP
    assert k < KAPPA_MAX, chain
    return k


def kappa_fma(chain):
    """A sequential fp32 fma chain of `chain` terms: gamma_chain = chain * u / (1 - chain * u)."""
    k = chain * U / (1 - chain * U)
    assert k < KAPPA_MAX, chain
    return k


def kappa_split(chain_main, chain_cross=None):
    """Split operands (edg_split.cu): x s = hi + lo to 2^-22 |x s| each, and the dropped lo x lo term is below
    2^-22 |a||b|, so the representation costs 3 * 2^-22; the hi x hi chain is a tcgen05 chain of `chain_main`, the
    cross terms (2^-11 smaller) one of `chain_cross`, and the epilogue adds the two accumulators (one u)."""
    k = 3 * 2.0 ** -22 + kappa_tc(chain_main) + 2 * 2.0 ** -11 * kappa_tc(chain_cross or chain_main) + U
    assert k < KAPPA_MAX
    return k


def split_floor(amax_a, amax_b, sum_abs_b, sum_abs_a):
    """Absolute floor of the split representation: lo is an fp16 subnormal below 2^-14, so each element also carries
    up to 2^-25 / s <= 2^-38 amax of absolute error."""
    return 2.0 ** -37 * (amax_a * sum_abs_b + amax_b * sum_abs_a)


# ------------------------------------------------------------------------------------------------ host rules
def pick_block_n(Nout, granule):
    """pick_block_n of edg_gemm_tc.cu -> (block_n, n_tiles)."""
    nt = cdiv(Nout, 256)
    bn = cdiv(cdiv(Nout, nt), granule) * granule
    if bn > 256:
        nt += 1
        bn = cdiv(cdiv(Nout, nt), granule) * granule
    return bn, cdiv(Nout, bn)


def linear_bf16_kernel(M, K, Nout):
    """Which kernel bf16 edg_linear runs (launch_linear_tc): the weight-stationary one when one N tile of the weight
    plus four activation stages fit in 227 KB and M >= 512."""
    bn, nt = pick_block_n(Nout, 16)
    w_bytes = cdiv(K, 64) * bn * 64 * 2
    fixed = 1024 + 1024 * 4 + 512
    return "ws" if (w_bytes + fixed + 4 * 128 * 64 * 2 <= 227 * 1024 and nt <= NUM_SMS and M >= 512) else "tc"


def odd16_multi_tile(Nout):
    bn, nt = pick_block_n(Nout, 16)
    return bn % 32 == 16 and nt > 1


def plan_linear_split(K, Nout):
    """plan_linear_split -> (ok, block_n, n_tiles)."""
    num_kb = cdiv(K, 64)
    fixed, budget = 1024 + 1024 * 4 + 512, 227 * 1024
    bn = 256
    while bn >= 16 and fixed + 2 * num_kb * bn * 64 * 2 + 2 * 2 * 128 * 64 * 2 > budget:
        bn -= 16
    bn = min(bn, 128)
    if bn < 16 or Nout > 1024:
        return False, 0, 0
    nt = cdiv(Nout, bn)
    block_n = cdiv(cdiv(Nout, nt), 16) * 16
    stages = min((budget - fixed - 2 * num_kb * block_n * 64 * 2) // (2 * 128 * 64 * 2), 8)
    return stages >= 2 and nt <= NUM_SMS, block_n, nt


F32_TC_MIN_ROWS = 1024


def linear_f32_kernel(M, K, Nout, out="f32"):
    """Which kernel ops.linear runs for fp32 operands."""
    if out == "f32" and M >= F32_TC_MIN_ROWS and plan_linear_split(K, Nout)[0]:
        return "split"
    if out == "f32" and M >= 512 and Nout >= 96 and K >= 32:       # big_linear_ok
        return "big"
    return "simt"


def plan_wgrad_tc(R, K1, K2, max_rows=0):
    bn, nt = pick_block_n(K2, 64)
    mt = cdiv(K1, 128)
    splits = max(min(cdiv(NUM_SMS, mt * nt), cdiv(R, 256)), 1)
    rows_per = cdiv(cdiv(R, splits), 64) * 64
    if max_rows and rows_per > max_rows:
        waves = cdiv(rows_per, max_rows)
        rows_per = cdiv(cdiv(R, splits * waves), 64) * 64
    return dict(block_n=bn, n_tiles=nt, m_tiles=mt, splits=max(cdiv(R, rows_per), 1), rows_per=rows_per)


def plan_wgrad_tall(R, K1e, K2e, max_rows=0):
    mt = cdiv(K1e, 128)
    ok = mt <= 3 and R >= 64 * NUM_SMS
    bn = 160
    while bn > 32 and bn - 32 >= K2e:
        bn -= 32
    ok = ok and mt * bn <= 512
    nt = cdiv(K2e, bn)
    want = max(NUM_SMS // nt, 1)
    rows_per = cdiv(cdiv(R, want), 64) * 64
    if max_rows and rows_per > max_rows:
        waves = cdiv(rows_per, max_rows)
        rows_per = cdiv(cdiv(R, want * waves), 64) * 64
    return dict(ok=ok, block_n=bn, n_tiles=nt, m_tiles=mt, splits=cdiv(R, rows_per), rows_per=rows_per)


K_SPLIT_MAIN_ROWS = 768


def wgrad_tc_plan(R, K1, K2, bias_of, max_rows=0):
    """(kernel, plan) of run_wgrad_tc for the extended shape."""
    K1e, K2e = K1 + (bias_of == 2), K2 + (bias_of == 1)
    t = plan_wgrad_tall(R, K1e, K2e, max_rows)
    if t["ok"]:
        return "tall", t
    return "tc", plan_wgrad_tc(R, K1e, K2e, max_rows)


def wgrad_f32_plan(R, K1, K2):
    """(kernel, rows per chain, slabs) of launch_wgrad_simt."""
    if R >= 4096 and K1 >= 96 and K2 >= 96:                         # big_wgrad_ok
        tiles = cdiv(K1, 128) * cdiv(K2, 128)
        sb = max(min(cdiv(4 * NUM_SMS, tiles), cdiv(R, 512)), 1)
        rp = cdiv(cdiv(R, sb), 8) * 8
        return "big", rp, cdiv(R, rp)
    tiles = cdiv(K1, 64) * cdiv(K2, 64)
    s = max(min(cdiv(4 * NUM_SMS, tiles), cdiv(R, 256)), 1)
    return "simt", cdiv(cdiv(R, s), 16) * 16, s


def wgrad_kappa(path, R, K1, K2, bias_of):
    """kappa of dW (and of the bias vector) for one edg_wgrad / edg_wgrad_split call: the longest chain of one CTA
    plus the partial-sum slabs the reduction adds (at most one u each)."""
    if path == "bf16":
        kind, p = wgrad_tc_plan(R, K1, K2, bias_of)
        k = kappa_tc(p["rows_per"]) + p["splits"] * U
        return k, k
    if path == "f32":
        kind, rp, slabs = wgrad_f32_plan(R, K1, K2)
        chunks = cdiv(R, 1024)
        return kappa_fma(rp + slabs), kappa_fma(min(R, 1024) // 8 + 8 + chunks + 1)   # edg_colsum: 8 row lanes
    _, main = wgrad_tc_plan(R, K1, K2, bias_of, K_SPLIT_MAIN_ROWS)
    _, cross = wgrad_tc_plan(R, K1, K2, bias_of)
    slabs = main["splits"] + 2 * cross["splits"]
    k = kappa_split(main["rows_per"], cross["rows_per"]) + slabs * U
    return k, k


# ------------------------------------------------------------------------------------------------ harness
def lib():
    from ed_gated_gcn_b200 import _lib
    return _lib.load()


def row_pitch(n, dt):
    return cdiv(n, 16 // (2 if dt == "bf16" else 4)) * (16 // (2 if dt == "bf16" else 4))


class Out:
    """A [rows, cols] output view of pitch `ld` inside a NaN-filled flat allocation: LEAD elements before row 0 and
    `guard` rows after the last.  `zero_to` = the columns up to which the kernel must zero the row padding."""

    def __init__(self, rows, cols, dt, ld=None, guard=1, zero_to=None):
        self.rows, self.cols, self.dt = rows, cols, dt
        self.ld = ld or row_pitch(cols, dt)
        self.zero_to = cols if zero_to is None else zero_to
        self.flat = torch.full(((rows + guard) * self.ld + 2 * LEAD,), NAN, dtype=TORCH_DT[dt], device=DEV)
        self.full = self.flat[LEAD:LEAD + rows * self.ld].view(rows, self.ld)
        self.view = self.full[:, :cols]

    def check_frame(self, what):
        """Row padding [cols, zero_to) exactly 0, everything outside the rows' first zero_to columns still NaN."""
        pad = self.full[:, self.cols:self.zero_to]
        assert bool((pad == 0).all()), f"{what}: row padding not zeroed"
        assert bool(self.full[:, self.zero_to:].isnan().all()), f"{what}: written past the row padding"
        assert bool(self.flat[:LEAD].isnan().all()), f"{what}: written before the first row"
        assert bool(self.flat[LEAD + self.rows * self.ld:].isnan().all()), f"{what}: written past the last row"

    def untouched(self):
        return bool(self.flat.isnan().all())


def vec_out(n):
    """A length-n fp32 vector inside NaN guards: (flat, view)."""
    flat = torch.full((n + 2 * LEAD,), NAN, dtype=torch.float32, device=DEV)
    return flat, flat[LEAD:LEAD + n]


def nan_padded(x, dt):
    """`x` (fp32, any device) as a device column slice of pitch row_pitch + one 16-byte chunk; the extra columns NaN."""
    R, C = x.shape
    ld = row_pitch(C, dt) + 16 // (2 if dt == "bf16" else 4)
    base = torch.full((max(R, 1), ld), NAN, dtype=TORCH_DT[dt], device=DEV)
    base[:R, :C] = x.to(device=DEV, dtype=TORCH_DT[dt])
    return base[:R, :C]


def scaled_rows(R, C, gen, span=8, scale=1.0):
    """randn rows times 2^e_r, e_r uniform in [-span, span]: exact in bf16 after rounding the randn part."""
    e = torch.randint(-span, span + 1, (R, 1), generator=gen).double()
    return (torch.randn(R, C, generator=gen).double() * torch.pow(2.0, e) * scale).float()


def bits(t):
    return t.contiguous().view(torch.int16 if t.element_size() == 2 else torch.int32)


def assert_within(got, want, bound, what, family):
    """|got - want| <= bound element-wise (NaN in got fails); records the worst ratio of `family`."""
    got = got.double()
    err = (got - want).abs()
    ok = err <= bound
    ratio = float((err / bound.clamp_min(1e-300)).nan_to_num(float("inf")).max()) if err.numel() else 0.0
    WORST[family] = max(WORST.get(family, 0.0), ratio)
    if not bool(ok.all()):
        idx = tuple(int(i) for i in torch.nonzero(~ok)[0])
        raise AssertionError(f"{what}: {int((~ok).sum())} elements out of bound, first {idx}: got {float(got[idx])!r} "
                             f"want {float(want[idx])!r} bound {float(bound[idx])!r} (worst ratio {ratio:.3g})")


@pytest.fixture(scope="module", autouse=True)
def _report_worst_ratios():
    yield
    if WORST:
        print("\nworst |err| / bound per family: " + ", ".join(f"{k} {v:.3g}" for k, v in sorted(WORST.items())))


def linear_expect(a, w, bias, act, out_dt, kappa, floor=None):
    """fp64 reference and bound of act(a w^T + bias) on the stored operands (device tensors)."""
    a64, w64 = a.double(), w.double()
    pre = a64 @ w64.t()
    S = a64.abs() @ w64.abs().t()
    b = bias.double() if bias is not None else torch.zeros(w.shape[0], dtype=torch.float64, device=DEV)
    pre_err = kappa * S + U * (S + b.abs()) + (floor if floor is not None else 0.0)
    pre = pre + b
    if act == 1:
        want, err = torch.sigmoid(pre), 0.25 * pre_err + ACT_ERR
    elif act == 2:
        want, err = pre.clamp_min(0), pre_err
    else:
        want, err = pre, pre_err
    if out_dt == "bf16":
        err = err + U_BF16 * (want.abs() + err)
    return want, err


def run_linear(a, w, bias, act, out_dt):
    """ops.linear into a NaN sentinel output of the ops row pitch."""
    from ed_gated_gcn_b200 import ops
    M, Nout = a.shape[0], w.shape[0]
    o = Out(M, Nout, out_dt, zero_to=row_pitch(Nout, out_dt))
    ops.linear(a, w, bias, act, out_dtype=TORCH_DT[out_dt], out=o.view)
    return o


def linear_inputs(M, K, Nout, dt, seed, a_scale=1.0):
    g = torch.Generator().manual_seed(seed)
    a = nan_padded(scaled_rows(M, K, g, scale=a_scale), dt)
    w = nan_padded(scaled_rows(Nout, K, g), dt)
    bias = (torch.randn(Nout, generator=g) * 4).to(DEV)
    return a, w, bias


# ------------------------------------------------------------------------------------------------ bf16 projection
NOUTS = (8, 16, 24, 34, 48, 200, 256, 257, 272, 288, 300, 320, 400, 520, 600, 768, 1000, 1024)
KS = (8, 16, 40, 63, 64, 65, 300, 768)
MS = (1, 127, 128, 129, 511, 512, 513, 20001)
K_PAST_WS = 1000            # at Nout = 300 the weight tile no longer fits: linear_tc at M >= 512


def bf16_linear_shapes():
    """Every Nout on both kernels (K rotating), the M and K sweeps, and the persistent shapes."""
    out = []
    for i, n in enumerate(NOUTS):
        out.append((129 if i % 2 else 300, KS[i % len(KS)], n))
        out.append((513 if i % 2 else 4096, KS[(i + 3) % len(KS)], n))
    out += [(m, 300, 272) for m in MS] + [(m, 65, 1000) for m in MS[:5]]
    out += [(513, k, 400) for k in KS] + [(129, k, 520) for k in KS]
    out += [(4096, K_PAST_WS, 300), (20001, 768, 400), (20001, 768, 768), (300, 300, 272), (4096, 300, 520)]
    seen, uniq = set(), []
    for s in out:
        if s not in seen:
            seen.add(s)
            uniq.append(s)
    return uniq


BF16_LINEAR = bf16_linear_shapes()


@pytest.mark.gpu
@pytest.mark.parametrize("out_dt", ["f32", "bf16"])
@pytest.mark.parametrize("shape", BF16_LINEAR, ids=[f"M{m}-K{k}-N{n}-{linear_bf16_kernel(m, k, n)}" for m, k, n in BF16_LINEAR])
def test_linear_bf16(shape, out_dt):
    M, K, Nout = shape
    i = BF16_LINEAR.index(shape)
    act, with_bias = i % 3, (i // 3) % 2 == 0
    a, w, bias = linear_inputs(M, K, Nout, "bf16", seed=i)
    bias = bias if with_bias else None
    o = run_linear(a, w, bias, act, out_dt)
    o.check_frame(f"{shape}")
    want, err = linear_expect(a, w, bias, act, out_dt, kappa_tc(K))
    assert_within(o.view, want, err, f"{shape} act {act} bias {with_bias}", f"linear_{linear_bf16_kernel(M, K, Nout)}_{out_dt}")


ODD16 = [(300, 300, 272), (513, 300, 272), (4096, 300, 520), (20001, 768, 400)]


@pytest.mark.gpu
@pytest.mark.parametrize("shape", ODD16, ids=[f"M{m}-K{k}-N{n}-{linear_bf16_kernel(m, k, n)}" for m, k, n in ODD16])
@pytest.mark.parametrize("out_dt", ["f32", "bf16"])
def test_linear_bf16_odd16_tiles_every_epilogue(shape, out_dt):
    """Both kernels at tiles that end inside their last 32-column chunk, with every activation and with / without
    bias: the chunk past the tile's end belongs to the next N tile."""
    M, K, Nout = shape
    assert odd16_multi_tile(Nout)
    a, w, bias = linear_inputs(M, K, Nout, "bf16", seed=M + Nout)
    for act in (0, 1, 2):
        for b in (bias, None):
            o = run_linear(a, w, b, act, out_dt)
            o.check_frame(f"{shape} act {act}")
            want, err = linear_expect(a, w, b, act, out_dt, kappa_tc(K))
            assert_within(o.view, want, err, f"{shape} act {act} bias {b is not None}",
                          f"linear_{linear_bf16_kernel(M, K, Nout)}_{out_dt}")


WS_BUDGET = [(513, 300, 272), (4096, 300, 520), (2048, 64, 1000), (112640, 300, 300)]


@pytest.mark.gpu
@pytest.mark.parametrize("shape", WS_BUDGET, ids=[f"M{m}-K{k}-N{n}" for m, k, n in WS_BUDGET])
def test_linear_ws_under_sm_budget_is_bitwise_the_unbudgeted_result(shape):
    """edg_set_sm_budget changes which CTA runs a tile, never a tile's sum: n = 1, 5, 74, 147 (at M = 112,640 and
    n = 5, 4 CTAs walk 440 M tiles each, wrapping both accumulator stages many times)."""
    from ed_gated_gcn_b200 import ops
    M, K, Nout = shape
    assert linear_bf16_kernel(M, K, Nout) == "ws"
    out_dt = "bf16" if M > 100000 else "f32"
    a, w, bias = linear_inputs(M, K, Nout, "bf16", seed=M)
    ref = run_linear(a, w, bias, 2, out_dt)
    ref.check_frame(f"{shape}")
    want, err = linear_expect(a, w, bias, 2, out_dt, kappa_tc(K))
    assert_within(ref.view, want, err, f"{shape}", f"linear_ws_{out_dt}")
    for n in (1, 5, 74, 147):
        with ops.sm_budget(n):
            o = run_linear(a, w, bias, 2, out_dt)
        assert torch.equal(bits(o.flat), bits(ref.flat)), f"{shape}: budget {n} changed the result"


def _edg_linear_rc(a, w, bias, o, out_dt, M=None):
    from ed_gated_gcn_b200 import _lib as L
    return lib().edg_linear(L.ptr(a), L.dt(a), a.stride(0), a.shape[0] if M is None else M, a.shape[1], L.ptr(w),
                            w.stride(0), w.shape[0], L.ptr(bias), 0, L.ptr(o.view), L.dt(TORCH_DT[out_dt]), o.ld,
                            L.stream())


@pytest.mark.gpu
@pytest.mark.parametrize("out_dt", ["f32", "bf16"])
def test_linear_bf16_refusals(out_dt):
    """bf16 Nout past 1024 has no N tile plan: refused, output untouched; M = 0 returns OK without writing."""
    for Nout in (1025, 1032):
        a, w, bias = linear_inputs(600, 64, Nout, "bf16", seed=Nout)
        o = Out(600, Nout, out_dt)
        assert _edg_linear_rc(a, w, bias, o, out_dt) == ERR["UNSUPPORTED"]
        torch.cuda.synchronize()
        assert o.untouched()
    a, w, bias = linear_inputs(4, 64, 300, "bf16", seed=0)
    o = Out(4, 300, out_dt)
    assert _edg_linear_rc(a, w, bias, o, out_dt, M=0) == ERR["OK"]
    torch.cuda.synchronize()
    assert o.untouched()


# ------------------------------------------------------------------------------------------------ fp32 projection
F32_LINEAR = [
    (511, 64, 128, "f32"), (512, 64, 128, "f32"),           # big_linear_ok: M
    (1023, 300, 300, "f32"), (1024, 300, 300, "f32"),       # F32_TC_MIN_ROWS
    (600, 64, 95, "f32"), (600, 64, 96, "f32"),             # big_linear_ok: Nout
    (600, 31, 128, "f32"), (600, 32, 128, "f32"),           # big_linear_ok: K
    (100, 37, 50, "f32"), (600, 301, 130, "f32"), (2048, 301, 300, "f32"),   # K % 4 != 0: load4's scalar tail
    (2048, 64, 1100, "f32"),                                # split refuses Nout > 1024: linear_big
    (1024, 768, 1024, "f32"), (1, 300, 300, "f32"), (4096, 128, 34, "f32"),
    (600, 300, 300, "bf16"), (2048, 301, 34, "bf16"),       # fp32 operands, bf16 output: linear_simt
]


def f32_kappa(kind, K):
    return kappa_split(K) if kind == "split" else kappa_fma(K)


def f32_floor(kind, a, w):
    if kind != "split":
        return None
    a64, w64 = a.double(), w.double()
    return split_floor(float(a64.abs().max()), float(w64.abs().max()), w64.abs().sum(1)[None, :], a64.abs().sum(1)[:, None])


@pytest.mark.gpu
@pytest.mark.parametrize("case", F32_LINEAR, ids=[f"M{m}-K{k}-N{n}-{o}-{linear_f32_kernel(m, k, n, o)}" for m, k, n, o in F32_LINEAR])
def test_linear_f32(case):
    M, K, Nout, out_dt = case
    kind = linear_f32_kernel(M, K, Nout, out_dt)
    i = F32_LINEAR.index(case)
    a, w, bias = linear_inputs(M, K, Nout, "f32", seed=100 + i)
    for act in (0, 1, 2):
        b = bias if act != 1 or i % 2 else None
        o = run_linear(a, w, b, act, out_dt)
        o.check_frame(f"{case} act {act}")
        want, err = linear_expect(a, w, b, act, out_dt, f32_kappa(kind, K), f32_floor(kind, a, w))
        assert_within(o.view, want, err, f"{case} act {act}", f"linear_{kind}_{out_dt}")


@pytest.mark.gpu
@pytest.mark.parametrize("edge", ["zero", "tiny", "huge", "wide_rows"])
@pytest.mark.parametrize("act", [0, 1, 2])
def test_linear_split_edges(edge, act):
    """The split path at the ends of its scale rule: an all-zero operand (amax = 0) gives exactly act(bias);
    operands scaled by 1e-30 and 1e30; rows whose magnitudes span e^N(0, 2) (what a per-tensor scale must survive)."""
    M, K, Nout = 2048, 300, 300
    assert linear_f32_kernel(M, K, Nout) == "split"
    g = torch.Generator().manual_seed(len(edge) + act)
    if edge == "wide_rows":
        x = torch.randn(M, K, generator=g) * torch.exp(2 * torch.randn(M, 1, generator=g))
    else:
        x = scaled_rows(M, K, g, scale={"zero": 0.0, "tiny": 1e-30, "huge": 1e30}[edge])
    a = nan_padded(x, "f32")
    w = nan_padded(scaled_rows(Nout, K, g), "f32")
    bias = (torch.randn(Nout, generator=g) * 4 * {"tiny": 1e-30, "huge": 1e30}.get(edge, 1.0)).to(DEV)
    o = run_linear(a, w, bias, act, "f32")
    o.check_frame(edge)
    if edge == "zero" and act != 1:
        want = bias.clamp_min(0) if act == 2 else bias
        assert torch.equal(o.view, want[None, :].expand(M, Nout)), "amax = 0 must give exactly act(bias)"
        return
    want, err = linear_expect(a, w, bias, act, "f32", kappa_split(K), f32_floor("split", a, w))
    assert_within(o.view, want, err, f"{edge} act {act}", "linear_split_f32")


# ------------------------------------------------------------------------------------------------ weight gradients
def wgrad_inputs(R, K1, K2, dt, seed):
    g = torch.Generator().manual_seed(seed)
    # scales on the columns of A and B: the rows of dW = A^T B and its columns
    a = (scaled_rows(K1, R, g).t() if R else torch.zeros(0, K1)).contiguous()
    b = (scaled_rows(K2, R, g).t() if R else torch.zeros(0, K2)).contiguous()
    return nan_padded(a, dt), nan_padded(b, dt)


def run_wgrad(path, a, b, bias_of, lddw_extra=0, accumulate=0, prefill=None):
    """edg_wgrad (path bf16 / f32) or edg_wgrad_split (path split) into NaN sentinels -> (Out dW, (flat, db))."""
    from ed_gated_gcn_b200 import _lib as L, ops
    R, K1 = a.shape
    K2 = b.shape[1]
    dW = Out(K1, K2, "f32", ld=K2 + lddw_extra)
    nb = K1 if bias_of == 1 else K2
    db = vec_out(nb)
    if prefill is not None:
        dW.view.copy_(prefill[0])
        db[1].copy_(prefill[1][:nb])
    dbp = L.ptr(db[1]) if bias_of else None
    if path == "split":
        sa, sb = ops.split_rows(a), ops.split_rows(b)
        n = lib().edg_wgrad_split_workspace(R, K1, K2)
        ws = torch.empty((n + 255) // 4, dtype=torch.float32, device=DEV)
        L.call("edg_wgrad_split", L.ptr(sa.data), sa.data.stride(0), L.ptr(sa.amax), K1, L.ptr(sb.data),
               sb.data.stride(0), L.ptr(sb.amax), K2, R, L.ptr(dW.view), dW.ld, dbp, bias_of, L.ptr(ws), ws.numel() * 4,
               L.stream())
    else:
        dt = L.dt(a)
        n = lib().edg_wgrad_workspace(R, K1, K2, dt)
        ws = torch.empty((n + 255) // 4, dtype=torch.float32, device=DEV)
        L.call("edg_wgrad", L.ptr(a), a.stride(0), K1, L.ptr(b), b.stride(0), K2, dt, R, L.ptr(dW.view), dW.ld, dbp,
               bias_of, accumulate, L.ptr(ws), ws.numel() * 4, L.stream())
    return dW, db


def check_wgrad(path, a, b, bias_of, dW, db, what, prefill=None):
    R, K1 = a.shape
    K2 = b.shape[1]
    dW.check_frame(what)
    a64, b64 = a.double(), b.double()
    kw, kb = wgrad_kappa(path, R, K1, K2, bias_of)
    want = a64.t() @ b64
    S = a64.abs().t() @ b64.abs()
    floor = 0.0
    if path == "split" and R:
        floor = split_floor(float(a64.abs().max()), float(b64.abs().max()), b64.abs().sum(0)[None, :],
                            a64.abs().sum(0)[:, None])
    err = kw * S + floor
    if prefill is not None:
        want = want + prefill[0].double()
        err = err + U * (want.abs() + prefill[0].double().abs())
    family = "wgrad_" + (wgrad_tc_plan(R, K1, K2, bias_of)[0] if path == "bf16" and R else path)
    assert_within(dW.view, want, err, what, family)
    flat, v = db
    assert bool(flat[:LEAD].isnan().all()) and bool(flat[LEAD + v.numel():].isnan().all()), f"{what}: db guards"
    if not bias_of:
        assert bool(v.isnan().all()), f"{what}: db written without bias_of"
        return
    x64 = a64 if bias_of == 1 else b64
    wb, Sb = x64.sum(0), x64.abs().sum(0)
    eb = kb * Sb
    if path == "split" and R:
        eb = eb + 2.0 ** -37 * float(x64.abs().max()) * R
    if prefill is not None:
        pb = prefill[1][:v.numel()].double()
        wb = wb + pb
        eb = eb + U * (wb.abs() + pb.abs())
    assert_within(v, wb, eb, what + " db", family + "_db")


R_SWEEP = (1, 63, 64, 65, 4095, 4096, 9471, 9472)
K1_SWEEP = (16, 127, 128, 129, 383, 384, 385)
K2_SWEEP = (24, 32, 33, 64, 65, 159, 160, 161, 300, 520, 1024)
BOX = (64, 128, 160, 256)


def wgrad_cases():
    """(path, R, K1, K2, bias_of): the R sweep on every path, K1 across the tall kernel's three-M-tile limit with the
    ones row (bias_of 2) planted at K1, K2 across the tall N tile steps with the ones column (bias_of 1), the ones on
    a box boundary and inside a partial last 64-row block, and the split path in waves of kSplitMainRows."""
    out = []
    for path in ("bf16", "f32"):
        out += [(path, R, 129, 161, bo) for R in R_SWEEP for bo in (0, 1, 2)]
    out += [("split", R, 129, 161, bo) for R in (1, 65, 4096, 9472) for bo in (0, 1, 2)]
    out += [("bf16", R, k1, 100, bo) for R in (4095, 9472) for k1 in K1_SWEEP for bo in (0, 2)]
    out += [("bf16", R, 96, k2, bo) for R in (1000, 9472) for k2 in K2_SWEEP for bo in (0, 1)]
    out += [("bf16", R, k, 96, 2) for R in (4095, 9500) for k in BOX] + [("bf16", R, 96, k, 1) for R in (4095, 9500) for k in BOX]
    out += [("f32", 4096, 95, 100, 1), ("f32", 4096, 96, 96, 2), ("f32", 4096, 301, 33, 2), ("f32", 5000, 300, 300, 1)]
    out += [("split", 2048, 300, 300, 1), ("split", 65536, 300, 300, 2), ("split", 4096, 385, 1024, 2),
            ("split", 9500, 160, 64, 1)]
    return out


WGRAD = wgrad_cases()


def _wgrad_id(c):
    path, R, K1, K2, bo = c
    kind = wgrad_tc_plan(R, K1, K2, bo)[0] if path == "bf16" else (wgrad_f32_plan(R, K1, K2)[0] if path == "f32" else "split")
    return f"{path}-R{R}-K1{K1}-K2{K2}-b{bo}-{kind}"


@pytest.mark.gpu
@pytest.mark.parametrize("case", WGRAD, ids=[_wgrad_id(c) for c in WGRAD])
def test_wgrad(case):
    path, R, K1, K2, bias_of = case
    a, b = wgrad_inputs(R, K1, K2, "f32" if path == "split" else path, seed=R + K1 + K2 + bias_of)
    dW, db = run_wgrad(path, a, b, bias_of)
    check_wgrad(path, a, b, bias_of, dW, db, str(case))
    dW2, db2 = run_wgrad(path, a, b, bias_of)
    assert torch.equal(bits(dW2.flat), bits(dW.flat)) and torch.equal(bits(db2[0]), bits(db[0])), f"{case}: not deterministic"


WGRAD_ABI = [("bf16", 4095, 129, 161), ("bf16", 9472, 384, 300), ("f32", 4096, 129, 161), ("f32", 300, 40, 33)]


@pytest.mark.gpu
@pytest.mark.parametrize("case", WGRAD_ABI, ids=[f"{p}-R{r}-K1{a}-K2{b}" for p, r, a, b in WGRAD_ABI])
@pytest.mark.parametrize("bias_of", [1, 2])
def test_wgrad_abi_accumulate_pitch_and_empty(case, bias_of):
    """accumulate = 1 onto known dW / db, a pitched dW (lddw > K2, extra columns stay NaN), and R = 0: zeros with
    accumulate 0, dW / db untouched with accumulate 1."""
    path, R, K1, K2 = case
    a, b = wgrad_inputs(R, K1, K2, path, seed=R + bias_of)
    g = torch.Generator().manual_seed(7)
    pre = ((torch.randn(K1, K2, generator=g) * 1e3).to(DEV), (torch.randn(max(K1, K2), generator=g) * 1e3).to(DEV))
    for extra in (0, 5):
        dW, db = run_wgrad(path, a, b, bias_of, lddw_extra=extra, accumulate=1, prefill=pre)
        check_wgrad(path, a, b, bias_of, dW, db, f"{case} accumulate lddw+{extra}", prefill=pre)
    e0, e1 = a[:0], b[:0]
    dW, db = run_wgrad(path, e0, e1, bias_of, lddw_extra=3)
    dW.check_frame("R = 0")
    assert bool((dW.view == 0).all()) and bool((db[1] == 0).all()), "R = 0, accumulate 0 must write zeros"
    dW, db = run_wgrad(path, e0, e1, bias_of, lddw_extra=3, accumulate=1, prefill=pre)
    torch.cuda.synchronize()
    assert torch.equal(dW.view, pre[0]) and torch.equal(db[1], pre[1][:db[1].numel()]), "R = 0, accumulate 1 wrote"
    assert bool(dW.full[:, K2:].isnan().all())


# ------------------------------------------------------------------------------------------------ edg_wgrad_batch
def run_wgrad_batch(a_list, b_list, bias_of, lddw):
    from ed_gated_gcn_b200 import _lib as L
    n = len(a_list)
    R, K1 = a_list[0].shape
    K2 = b_list[0].shape[1]
    outs = [Out(K1, K2, "f32", ld=lddw) for _ in range(n)]
    dbs = [vec_out(K1 if bias_of == 1 else K2) for _ in range(n)]
    nbytes = lib().edg_wgrad_batch_workspace(n, R, K1, K2)
    ws = torch.empty((nbytes + 255) // 4, dtype=torch.float32, device=DEV)
    P = ctypes.c_void_p * n
    rc = lib().edg_wgrad_batch(n, P(*[L.ptr(a) for a in a_list]), a_list[0].stride(0), K1, P(*[L.ptr(b) for b in b_list]),
                               b_list[0].stride(0), K2, L.dt(a_list[0]), R, P(*[L.ptr(o.view) for o in outs]), lddw,
                               P(*[L.ptr(d[1]) for d in dbs]) if bias_of else None, bias_of, L.ptr(ws), ws.numel() * 4,
                               L.stream())
    return rc, outs, dbs


@pytest.mark.gpu
@pytest.mark.parametrize("n", range(1, 9))
@pytest.mark.parametrize("bias_of", [0, 1, 2])
def test_wgrad_batch(n, bias_of):
    """n problems with their own inputs, each against its own fp64 reference: a mixed-up map, slab or output
    pointer fails."""
    R, K1, K2 = 1000 + 37 * n, 129, 161
    ins = [wgrad_inputs(R, K1, K2, "bf16", seed=100 * n + i) for i in range(n)]
    rc, outs, dbs = run_wgrad_batch([x[0] for x in ins], [x[1] for x in ins], bias_of, K2 + 3)
    assert rc == ERR["OK"]
    p = plan_wgrad_tc(R, K1 + (bias_of == 2), K2 + (bias_of == 1))
    splits = max(min(cdiv(NUM_SMS, p["m_tiles"] * p["n_tiles"] * n), p["splits"]), 1)
    rows_per = cdiv(cdiv(R, splits), 64) * 64
    k = kappa_tc(rows_per) + cdiv(R, rows_per) * U
    for i, ((a, b), dW, db) in enumerate(zip(ins, outs, dbs)):
        dW.check_frame(f"problem {i}")
        a64, b64 = a.double(), b.double()
        assert_within(dW.view, a64.t() @ b64, k * (a64.abs().t() @ b64.abs()), f"n {n} problem {i}", "wgrad_batch")
        if bias_of:
            x = a64 if bias_of == 1 else b64
            assert_within(db[1], x.sum(0), k * x.abs().sum(0), f"n {n} problem {i} db", "wgrad_batch_db")


@pytest.mark.gpu
def test_wgrad_batch_refusals():
    a, b = wgrad_inputs(300, 64, 64, "bf16", seed=1)
    rc, outs, _ = run_wgrad_batch([a] * 9, [b] * 9, 0, 64)
    assert rc == ERR["UNSUPPORTED"]
    af, bf = wgrad_inputs(300, 64, 64, "f32", seed=1)
    rc2, outs2, _ = run_wgrad_batch([af] * 2, [bf] * 2, 0, 64)
    assert rc2 == ERR["DTYPE"]
    torch.cuda.synchronize()
    assert all(o.untouched() for o in outs + outs2)


# ------------------------------------------------------------------------------------------------ edg_mlp_chain
def chain_call(mode, a0_list, stages, M, D):
    """edg_mlp_chain through the C ABI -> status.  stages[g][s] = dict(w, bias, y, out (Out or None))."""
    from ed_gated_gcn_b200 import _lib as L
    G, S = len(a0_list), len(stages[0])
    arr = (L.ChainStage * (G * S))()
    for g in range(G):
        for s, st in enumerate(stages[g]):
            e = arr[g * S + s]
            e.w, e.ldw = L.ptr(st["w"]), st["w"].stride(0)
            e.bias = L.ptr(st.get("bias"))
            y = st.get("y")
            e.y, e.ldy = (L.ptr(y), y.stride(0)) if y is not None else (None, 0)
            o = st.get("out")
            e.out, e.ldo = (L.ptr(o.view), o.ld) if o is not None else (None, 0)
            e.out_dtype = L.dt(TORCH_DT[o.dt]) if o is not None else 0
    P = ctypes.c_void_p * G
    return lib().edg_mlp_chain(mode, G, S, P(*[L.ptr(a) for a in a0_list]), a0_list[0].stride(0), arr, M, D, L.stream())


def chain_case(mode, G, S, M, D, seed, out_dts=None, null_bias=False, null_y=False):
    g = torch.Generator().manual_seed(seed)
    a0 = [nan_padded(torch.rand(M, D, generator=g) if mode == 0 else scaled_rows(M, D, g, span=4), "bf16")
          for _ in range(G)]
    stages = []
    for k in range(G):
        st = []
        for s in range(S):
            w = nan_padded(scaled_rows(D, D, g, span=2) / D ** 0.5, "bf16")
            dt = (out_dts or ["bf16"] * S)[s]
            d = dict(w=w, out=Out(M, D, dt, zero_to=row_pitch(D, dt)))
            if mode == 0 and not (null_bias and (k + s) % 2 == 0):
                d["bias"] = torch.randn(D, generator=g).to(DEV)
            if mode == 1 and not (null_y and (k + s) % 2 == 0):
                d["y"] = nan_padded(torch.rand(M, D, generator=g), "bf16")
            st.append(d)
        stages.append(st)
    return a0, stages


def check_chain(mode, a0, stages, D, what):
    """Stage by stage on the stored operands: stage s + 1 reads the bf16 rounding of stage s's output, which is
    what the kernel writes back into its shared-memory tile (the stored bf16 output, or the fp32 one rounded)."""
    for k, st in enumerate(stages):
        x = a0[k].double()
        for s, d in enumerate(st):
            o = d["out"]
            o.check_frame(f"{what} group {k} stage {s}")
            w = d["w"].double()
            z, S = x @ w.t(), x.abs() @ w.abs().t()
            zerr = kappa_tc(D) * S
            if mode == 0:
                b = d["bias"].double() if d.get("bias") is not None else torch.zeros(D, dtype=torch.float64, device=DEV)
                want, err = torch.sigmoid(z + b), 0.25 * (zerr + U * (S + b.abs())) + ACT_ERR
            elif d.get("y") is not None:
                y = d["y"].double()
                want, err = z * y * (1 - y), zerr * y * (1 - y) + 3 * U * (z * y * (1 - y)).abs()
            else:
                want, err = z, zerr
            if o.dt == "bf16":
                err = err + U_BF16 * (want.abs() + err)
            assert_within(o.view, want, err, f"{what} group {k} stage {s}", f"mlp_chain_mode{mode}_{o.dt}")
            x = o.view.to(torch.bfloat16).double()


CHAIN = [(mode, G, S, D, M) for mode in (0, 1) for G in (1, 4) for S in (1, 3) for D in (16, 20, 312, 320)
         for M in ((1, 129) if D in (16, 320) else (200,))]


@pytest.mark.gpu
@pytest.mark.parametrize("case", CHAIN, ids=[f"mode{m}-G{g}-S{s}-D{d}-M{r}" for m, g, s, d, r in CHAIN])
def test_mlp_chain(case):
    mode, G, S, D, M = case
    out_dts = [("f32" if (s + D) % 2 == 0 and D % 4 == 0 else "bf16") for s in range(S)]
    a0, stages = chain_case(mode, G, S, M, D, seed=sum(case), out_dts=out_dts, null_bias=True, null_y=True)
    assert chain_call(mode, a0, stages, M, D) == ERR["OK"]
    check_chain(mode, a0, stages, D, str(case))


@pytest.mark.gpu
@pytest.mark.parametrize("bad", ["D15", "D321", "groups5", "stages4", "f32_out_D18"])
def test_mlp_chain_refusals(bad):
    G, S, D, out_dts = {"D15": (1, 2, 15, None), "D321": (1, 2, 321, None), "groups5": (5, 2, 64, None),
                        "stages4": (1, 4, 64, None), "f32_out_D18": (2, 2, 18, ["bf16", "f32"])}[bad]
    a0, stages = chain_case(0, G, S, 130, D, seed=3, out_dts=out_dts)
    assert chain_call(0, a0, stages, 130, D) == ERR["UNSUPPORTED"]
    torch.cuda.synchronize()
    assert all(d["out"].untouched() for st in stages for d in st)


# ------------------------------------------------------------------------------------------------ casts, colsum
def cast_source(R, C, seed):
    """fp32 values with bf16 rounding ties (both parities), subnormals, infinities and large values."""
    g = torch.Generator().manual_seed(seed)
    x = scaled_rows(R, C, g, span=20)
    flat = x.view(-1)
    n = flat.numel()
    special = torch.tensor([1 + 2 ** -8, 1 + 3 * 2 ** -8, -(1 + 2 ** -8), 2 ** -130, -2 ** -140, float("inf"),
                            -float("inf"), 3.3e38, 0.0, -0.0], dtype=torch.float32)
    flat[torch.arange(0, n, max(n // 10, 1))[:10]] = special[:min(10, n)]
    return x


@pytest.mark.gpu
@pytest.mark.parametrize("dst", ["bf16", "f32"])
@pytest.mark.parametrize("shape", [(1, 1), (7, 33), (300, 300), (129, 1000), (1025, 17)])
@pytest.mark.parametrize("transpose", [0, 1])
def test_cast_2d_is_torch_round_to_nearest(shape, transpose, dst):
    from ed_gated_gcn_b200 import _lib as L
    R, C = shape
    src = nan_padded(cast_source(R, C, R * C), "f32")
    ro, co = (C, R) if transpose else (R, C)
    o = Out(ro, co, dst, ld=row_pitch(co, dst) + 8)          # the kernel writes every column up to ldd
    L.call("edg_cast_2d", L.ptr(src), src.stride(0), R, C, L.ptr(o.view), L.dt(TORCH_DT[dst]), o.ld, transpose,
           L.stream())
    o.zero_to = o.ld
    o.check_frame(f"{shape}")
    want = (src.t() if transpose else src).to(TORCH_DT[dst])
    assert torch.equal(bits(o.view), bits(want))


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 32, 33, 45])
def test_cast_batch_is_torch_round_to_nearest(n):
    """edg_cast_batch directly (at most 32 items per launch: 33 are refused) and through ops.cast_weights_batch,
    which splits 33 or more items into two launches."""
    from ed_gated_gcn_b200 import _lib as L, ops
    shapes = [(1 + (7 * i) % 41, 1 + (13 * i) % 300) for i in range(n)]
    trs = [i % 2 for i in range(n)]
    srcs = [nan_padded(cast_source(r, c, i), "f32") for i, (r, c) in enumerate(shapes)]
    outs = [Out(c if t else r, r if t else c, "bf16") for (r, c), t in zip(shapes, trs)]
    for o in outs:
        o.zero_to = o.ld
    def arrays(sl):
        k = len(range(n)[sl])
        P, I32, I64 = ctypes.c_void_p * k, ctypes.c_int32 * k, ctypes.c_int64 * k
        return (k, P(*[L.ptr(s) for s in srcs[sl]]), P(*[L.ptr(o.view) for o in outs[sl]]), I32(*[r for r, _ in shapes[sl]]),
                I32(*[c for _, c in shapes[sl]]), I64(*[s.stride(0) for s in srcs[sl]]), I64(*[o.ld for o in outs[sl]]),
                I32(*trs[sl]))
    if n > 32:
        assert lib().edg_cast_batch(*arrays(slice(0, n)), L.BF16, L.stream()) == ERR["UNSUPPORTED"]
        torch.cuda.synchronize()
        assert all(o.untouched() for o in outs)
    for i0 in range(0, n, 32):
        assert lib().edg_cast_batch(*arrays(slice(i0, i0 + 32)), L.BF16, L.stream()) == ERR["OK"]
    for i, (s, o, t) in enumerate(zip(srcs, outs, trs)):
        o.check_frame(f"item {i}")
        assert torch.equal(bits(o.view), bits((s.t() if t else s).to(torch.bfloat16))), f"item {i}"
    got = ops.cast_weights_batch([(s.contiguous(), bool(t)) for s, t in zip(srcs, trs)], torch.bfloat16)
    for i, (s, o, t) in enumerate(zip(srcs, got, trs)):
        assert torch.equal(bits(o), bits((s.t() if t else s).to(torch.bfloat16))), f"ops item {i}"


@pytest.mark.gpu
@pytest.mark.parametrize("dt", ["bf16", "f32"])
@pytest.mark.parametrize("R", [0, 1, 1023, 1024, 1025, 5000])
@pytest.mark.parametrize("C", [1, 33, 300])
def test_colsum(dt, R, C):
    from ed_gated_gcn_b200 import _lib as L
    g = torch.Generator().manual_seed(R + C)
    x = nan_padded(scaled_rows(C, R, g).t().contiguous() if R else torch.zeros(0, C), dt)
    pre = (torch.randn(C, generator=g) * 100).to(DEV)
    chunks = cdiv(R, 1024)
    k = kappa_fma(min(R, 1024) // 8 + 8 + chunks + 1)
    x64 = x.double()
    for acc in (0, 1):
        flat, out = vec_out(C)
        if acc:
            out.copy_(pre)
        nbytes = lib().edg_colsum_workspace(R, C)
        ws = torch.empty(max(nbytes // 4, 1), dtype=torch.float32, device=DEV)
        L.call("edg_colsum", L.ptr(x), L.dt(x), x.stride(0), R, C, L.ptr(out), acc, L.ptr(ws), ws.numel() * 4, L.stream())
        want = x64.sum(0) + (pre.double() if acc else 0)
        err = k * x64.abs().sum(0) + (U * (want.abs() + pre.double().abs()) if acc else 0)
        assert_within(out, want, err, f"R {R} C {C} acc {acc}", "colsum")
        assert bool(flat[:LEAD].isnan().all()) and bool(flat[LEAD + C:].isnan().all())


# ------------------------------------------------------------------------------------------------ CPU-only
def _cpu_gemm_fp32(a, w, order):
    """fp32 C = a w^T summed sequentially over k in `order`, every product and sum rounded to fp32."""
    acc = torch.zeros(a.shape[0], w.shape[0], dtype=torch.float32)
    for k in order:
        acc = acc + a[:, k:k + 1] * w[:, k][None, :]
    return acc


def _within(got, want, bound):
    return bool(((got.double() - want).abs() <= bound).all())


def test_bounds_accept_a_shuffled_fp32_gemm_and_reject_a_dropped_k_step_or_a_neighbour_column():
    g = torch.Generator().manual_seed(5)
    M, K, Nout = 64, 300, 40
    a, w = scaled_rows(M, K, g), scaled_rows(Nout, K, g)
    a64, w64 = a.double(), w.double()
    want, S = a64 @ w64.t(), a64.abs() @ w64.abs().t()
    bound = kappa_fma(K) * S
    order = torch.randperm(K, generator=g).tolist()
    got = _cpu_gemm_fp32(a, w, order)
    assert _within(got, want, bound)
    for k0 in (0, 128, 288):                                  # one 16-wide k step left out
        dropped = _cpu_gemm_fp32(a, w, [k for k in order if not k0 <= k < k0 + 16])
        assert not _within(dropped, want, bound), k0
    for j in (0, 17, Nout - 2):                               # one column taken from its neighbour
        nb = got.clone()
        nb[:, j] = got[:, j + 1]
        assert not _within(nb, want, bound), j
    # the tensor-core and split models are tighter than the fp32 one and below 2^-14 at every chain the file uses
    assert kappa_tc(K) < kappa_fma(K) and kappa_split(K) < KAPPA_MAX


def test_host_rules_land_the_shapes_on_both_sides():
    # pick_block_n: the odd-16 widths of the issue, and how many of 1..1024 end a tile inside a 32-column chunk
    assert [pick_block_n(n, 16) for n in (257, 272, 400, 520, 600)] == [(144, 2), (144, 2), (208, 2), (176, 3), (208, 3)]
    assert sum(odd16_multi_tile(n) for n in range(1, 1025)) == 368
    assert {n for n in NOUTS if odd16_multi_tile(n)} == {257, 272, 288, 400, 520, 600}
    assert [pick_block_n(n, 16)[1] for n in (200, 256, 1000, 1024)] == [1, 1, 4, 4]
    # both bf16 kernels at odd-16 widths; the persistent linear_tc shape; the weight past the resident limit
    assert linear_bf16_kernel(300, 300, 272) == "tc"
    assert linear_bf16_kernel(513, 300, 272) == "ws" and linear_bf16_kernel(4096, 300, 520) == "ws"
    assert linear_bf16_kernel(511, 300, 272) == "tc" and linear_bf16_kernel(512, 300, 272) == "ws"
    assert linear_bf16_kernel(4096, K_PAST_WS, 300) == "tc" and linear_bf16_kernel(4096, 448, 300) == "ws"
    assert cdiv(20001, 128) * pick_block_n(400, 16)[1] == 314 and linear_bf16_kernel(20001, 768, 400) == "tc"
    assert cdiv(20001, 128) * pick_block_n(768, 16)[1] > 2 * NUM_SMS
    kinds = {linear_bf16_kernel(*s) for s in BF16_LINEAR}
    assert kinds == {"tc", "ws"}
    assert {linear_bf16_kernel(*s) for s in BF16_LINEAR if odd16_multi_tile(s[2])} == {"tc", "ws"}
    assert set(NOUTS) <= {s[2] for s in BF16_LINEAR} and set(KS) <= {s[1] for s in BF16_LINEAR}
    assert set(MS) <= {s[0] for s in BF16_LINEAR}
    # sm budget: at M = 112,640 and n = 5, 2 CTAs per N tile walk 440 M tiles each
    bn, nt = pick_block_n(300, 16)
    assert nt == 2 and (5 // nt) * nt == 4 and cdiv(112640, 128) // (5 // nt) == 440
    assert all(linear_bf16_kernel(*s) == "ws" for s in WS_BUDGET)
    # fp32: each side of big_linear_ok, F32_TC_MIN_ROWS and the split plan
    kind = {c: linear_f32_kernel(*c) for c in [c[:3] for c in F32_LINEAR]}
    assert kind[(511, 64, 128)] == "simt" and kind[(512, 64, 128)] == "big"
    assert kind[(1023, 300, 300)] == "big" and kind[(1024, 300, 300)] == "split"
    assert kind[(600, 64, 95)] == "simt" and kind[(600, 64, 96)] == "big"
    assert kind[(600, 31, 128)] == "simt" and kind[(600, 32, 128)] == "big"
    assert not plan_linear_split(64, 1100)[0] and kind[(2048, 64, 1100)] == "big"
    assert {k for k in kind.values()} == {"simt", "big", "split"}
    assert any(c[1] % 4 and linear_f32_kernel(*c[:3]) == k for c in F32_LINEAR for k in ("simt", "big", "split"))
    # weight gradients: the tall threshold in R and in K1e, the tall N tile steps, the big FFMA kernel, the waves
    assert wgrad_tc_plan(9471, 129, 161, 0)[0] == "tc" and wgrad_tc_plan(9472, 129, 161, 0)[0] == "tall"
    assert wgrad_tc_plan(9472, 384, 100, 0)[0] == "tall" and wgrad_tc_plan(9472, 384, 100, 2)[0] == "tc"
    assert wgrad_tc_plan(9472, 383, 100, 2)[0] == "tall" and wgrad_tc_plan(9472, 385, 100, 0)[0] == "tc"
    tall_bn = {k2: wgrad_tc_plan(9472, 96, k2, 1)[1]["block_n"] for k2 in K2_SWEEP}
    assert {tall_bn[k] for k in (24, 32, 33, 64, 65, 159, 160)} == {32, 64, 96, 160} and tall_bn[161] == 160
    assert {pick_block_n(k2, 64) for k2 in K2_SWEEP} >= {(64, 1), (192, 2), (256, 4)}
    assert wgrad_f32_plan(4095, 129, 161)[0] == "simt" and wgrad_f32_plan(4096, 129, 161)[0] == "big"
    assert wgrad_f32_plan(4096, 95, 100)[0] == "simt"
    full = plan_wgrad_tall(65536, 301, 300)
    waved = plan_wgrad_tall(65536, 301, 300, K_SPLIT_MAIN_ROWS)
    assert full["rows_per"] > K_SPLIT_MAIN_ROWS >= waved["rows_per"] and waved["splits"] > full["splits"]
    # the planted ones row / column on a box boundary and inside a partial last 64-row block
    assert {c[2] for c in WGRAD if c[4] == 2} >= set(BOX) and {c[3] for c in WGRAD if c[4] == 1} >= set(BOX)
    assert any(c[1] % 64 and c[4] and wgrad_tc_plan(*c[1:])[0] == "tall" for c in WGRAD if c[0] == "bf16")
    # every chain the file bounds stays below 2^-14 (the kappa helpers assert it)
    for c in WGRAD:
        if c[1]:
            wgrad_kappa(c[0], *c[1:])
