"""The row-streaming kernels of the gated block -- edg_pool_fwd, edg_scores_kl_fwd, edg_head_bwd -- and
edg_aggregate, each in both of its implementations, against fp64 references of the formulas in include/edgcn.h.

Each kernel has a window-staged implementation (edg_block_staged.cu: one bulk async copy of the rows of the sentences
that start in a window of `tile_rows` packed rows, sized by plan_window in edg_staged.cuh) and a per-sentence one
(edg_block.cu).  Host rules pick one per call from D, the dtype and max_len.  Every case here runs on the graph from
build_graph (staged wherever the rules allow) and on a copy with ``row_sent=None``, which the header documents as
"do not stage" (for edg_aggregate: the flat kernel).  The rules and plan_window are restated below; the layouts are
chosen with the restatement, and each asserts the geometry it is meant to have:
  - empty sentences before the first row, right after a sentence longer than a window (on a window's first row and
    at the end of the batch), inside and at the end of windows, and a batch with no rows at all;
  - sentences that straddle windows, runs of 1-token sentences, and for the scores kernel (lane = row, four passes of
    32 rows) lengths 31/32/33, 96/97, 128/129;
  - max_len at the last 72 KB plan, the first 200 KB plan, the last staged value and the first per-sentence value.
Every output is filled with a sentinel (NaN, or -7 for `arg`) before the kernel runs, so an element that no block
writes fails deterministically."""
import dataclasses

import numpy as np
import pytest
import torch

from gpu_util import DEV
from test_gpu_g_fused_limits import adj_hat, assert_rows_close

pytestmark = pytest.mark.gpu

U = 2.0 ** -24                 # unit roundoff of fp32
U_BF16 = 2.0 ** -8             # unit roundoff of bf16 (8 significant bits)
ESIZE = {"bf16": 2, "f32": 4}
TORCH_DT = {"bf16": torch.bfloat16, "f32": torch.float32}
MAX_GRAPH_SENTENCE = 4096      # longest sentence build_graph / tree_distance take (kMaxSentence in edg_graph.cu)


# ------------------------------------------------------------------------------------------------ the host rules
def plan_window(pitch, max_len, extra=0, fixed=0):
    """plan_window of edg_staged.cuh -> (tile_rows, cap_rows, on the 200 KB plan)."""
    for big, budget in ((False, 72 * 1024), (True, 200 * 1024)):
        cap = (budget - fixed) // (pitch + extra) if budget > fixed else 0
        tile = cap - max_len + 1
        if tile >= 16 or big:
            return tile, cap, big


def geometry(kind, dt, D):
    """(16-byte chunks, row pitch in bytes, per-row extra, fixed extra) of a launcher's window."""
    E = 16 // ESIZE[dt]
    chunks = -(-D // E)
    pitch = chunks * 16
    if kind == "scores":
        return chunks, pitch, 0, 4 * chunks * E * 4           # per-warp gate*v of kScoresWarps = 4 warps
    return chunks, pitch, (4 if kind == "head" else 0), 0  # head: the ds row


def staged_plan(kind, dt, D, max_len, n_rows=1):
    """The launchers' decline rules (edg_block_staged.cu): the plan the staged kernel runs, or None when the
    per-sentence kernel runs."""
    chunks, pitch, extra, fixed = geometry(kind, dt, D)
    if max_len <= 0 or n_rows <= 0 or chunks > 256:
        return None
    if kind == "scores" and (chunks > 128 or max_len > 128):
        return None
    if kind == "head":
        y = max(1, min(8, 256 // chunks))
        if chunks * y < 32:                                    # phase 1 needs one full warp
            return None
    p = plan_window(pitch, max_len, extra, fixed)
    return p if p[0] >= 8 else None


def plan_points(kind, dt, D):
    """max_len at the last 72 KB plan, the first 200 KB plan, the last staged value, the first per-sentence value
    (those that exist for the shape)."""
    ms = [M for M in range(1, 8192) if staged_plan(kind, dt, D, M)]
    if not ms:
        return {}
    assert ms == list(range(1, ms[-1] + 1))                    # staged exactly for max_len 1 .. last
    small = [M for M in ms if not staged_plan(kind, dt, D, M)[2]]
    big = [M for M in ms if staged_plan(kind, dt, D, M)[2]]
    out = {"staged_last": ms[-1], "per_sentence_first": ms[-1] + 1}
    if small:
        out["plan72_last"] = small[-1]
    if big:
        out["plan200_first"] = big[0]
    return out


def parent_windows(lens, tile):
    """(r0, r1, s0, s1) of every window as stage_window computed them before every sentence had an owner: window w
    owned sentences s0 .. s1 - 1 and returned early when r1 <= r0.  Used to show what each layout exercises."""
    sp = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    B, N = len(lens), int(sp[-1])
    row_sent = np.repeat(np.arange(B), lens)
    out = []
    for w0 in range(0, N, tile):
        w1 = w0 + tile
        a0 = row_sent[w0] if w0 < N else B
        a1 = row_sent[w1] if w1 < N else B
        up0, up1 = w0 < N and sp[a0] < w0, w1 < N and sp[a1] < w1
        out.append((sp[a0 + 1] if up0 else sp[a0], sp[a1 + 1] if up1 else sp[a1], a0 + up0, a1 + up1))
    return out


def unowned_before_the_fix(lens, tile):
    """Sentences that no window with rows owned before the fix."""
    owned = np.zeros(len(lens), dtype=bool)
    for r0, r1, s0, s1 in parent_windows(lens, tile):
        if r1 > r0:
            owned[s0:s1] = True
    return set(np.nonzero(~owned)[0].tolist())


# ------------------------------------------------------------------------------------------------ layouts
BASE_LAYOUTS = ("lead1", "lead3", "empty_at_window_start", "empty_at_end_after_long", "empty_inside_windows",
                "all_empty", "straddle", "ones")
POINT_LAYOUTS = ("plan72_last", "plan200_first", "staged_last", "per_sentence_first")
SCORES_LAYOUTS = ("len31_32_33", "len96_97", "len128_129")
EMPTY_OWNER_LAYOUTS = ("lead1", "lead3", "empty_at_window_start", "empty_at_end_after_long", "all_empty")


def _fill(rng, lens, M, rows, lo=1):
    while sum(lens) < rows:
        lens.append(int(rng.integers(lo, M + 1)))
    return lens


def make_layout(kind, dt, D, name, seed):
    """(lengths, max_len, tile_rows of the staged kernel or None).  Asserts the layout's geometry wherever the staged
    kernel runs."""
    rng = np.random.default_rng(seed)
    pts = plan_points(kind, dt, D)
    if name in POINT_LAYOUTS:
        M = pts[name]
        p = staged_plan(kind, dt, D, M)
        nxt = staged_plan(kind, dt, D, M + 1)
        if name == "plan72_last":
            assert not p[2] and p[0] >= 16 and (nxt is None or nxt[2])
        elif name == "plan200_first":
            assert p[2] and not staged_plan(kind, dt, D, M - 1)[2]
        elif name == "staged_last":
            assert p is not None and nxt is None
        else:
            assert p is None and staged_plan(kind, dt, D, M - 1) is not None
        tile = p[0] if p else 8
        lens = _fill(rng, [M, 1], M, max(3 * tile, 3 * M))
        lens.append(M)
        return lens, M, (p[0] if p else None)
    if name in SCORES_LAYOUTS:
        base = {"len31_32_33": [31, 32, 33], "len96_97": [96, 97], "len128_129": [128, 129]}[name]
        lens = []
        for n in base:
            lens += [n, int(rng.integers(1, 30))]
        lens = base + lens
        M = max(lens)
        p = staged_plan(kind, dt, D, M)
        return lens, M, (p[0] if p else None)
    # base layouts: a moderate max_len; the ones that need a sentence spanning windows take the smallest max_len at
    # which the staged kernel has a sentence of at least two windows (2 * tile_rows <= max_len)
    staged = [M for M in range(1, 8192) if staged_plan(kind, dt, D, M)]
    M = min(48, staged[-1]) if staged else 48
    reachable = True
    if name in ("empty_at_window_start", "empty_at_end_after_long"):
        long_ok = [m for m in staged if 2 * staged_plan(kind, dt, D, m)[0] <= m]
        # (none for the scores kernel at small D: max_len <= 128 leaves windows longer than any sentence)
        reachable = bool(long_ok)
        M = long_ok[0] if long_ok else M
    p = staged_plan(kind, dt, D, M)
    tile = p[0] if p and reachable else 16
    if name == "lead1":
        lens = _fill(rng, [0], M, 3 * tile)
    elif name == "lead3":
        lens = _fill(rng, [0, 0, 0], M, 3 * tile)
    elif name == "empty_at_window_start":
        L = (M // tile) * tile                       # ends on a window start; the window before lies inside it
        lens = _fill(rng, [L, 0, 0, 5], M, L + 2 * tile)
    elif name == "empty_at_end_after_long":
        lens = _fill(rng, [3, 1], M, 2 * tile) + [min(M, 2 * tile), 0, 0]
    elif name == "empty_inside_windows":
        # every window holds whole short sentences, an empty one after the first (inside the window), some more at
        # random, and one after the last (on the boundary: the window that ends there owns it)
        lens, m = [], min(M, tile)
        for _ in range(4):
            left = tile
            while left:
                n = min(left, min(m, tile // 2) if left == tile else int(rng.integers(1, m + 1)))
                left -= n
                lens += [n, 0] if (left == tile - n or left == 0 or rng.random() < 0.3) else [n]
    elif name == "all_empty":
        lens = [0] * 7
    elif name == "straddle":
        lens = _fill(rng, [], M, 4 * tile, lo=max(1, min(M, tile) // 2))
        lens.append(M)
    elif name == "ones":
        lens = [1] * (3 * tile + 1) + [M] + [1] * 5
    else:
        raise ValueError(name)
    assert max(lens) <= M
    tile_staged = p[0] if p and sum(lens) > 0 else None
    if tile_staged and reachable:
        check_geometry(name, lens, tile_staged)
    return lens, M, tile_staged


def check_geometry(name, lens, tile):
    sp = np.concatenate([[0], np.cumsum(lens)])
    lost = unowned_before_the_fix(lens, tile)
    empty = [s for s, n in enumerate(lens) if n == 0]
    if name in ("lead1", "lead3"):
        k = 1 if name == "lead1" else 3
        assert parent_windows(lens, tile)[0][2] == k and lost == set(range(k))
    elif name == "empty_at_window_start":
        # sentences 1 and 2 are empty, start on a window's first row after a sentence longer than two windows, and
        # the window before them has no row to stage
        assert lens[0] >= 2 * tile and sp[1] % tile == 0 and lost == {1, 2}
    elif name == "empty_at_end_after_long":
        B = len(lens)
        assert lens[-3] > tile and lost == {B - 2, B - 1}
    elif name == "empty_inside_windows":
        assert not lost and any(sp[s] % tile == 0 for s in empty) and any(sp[s] % tile for s in empty)
    elif name == "straddle":
        assert any(sp[s] // tile != (sp[s + 1] - 1) // tile for s in range(len(lens)) if lens[s])
    elif name == "ones":
        assert lens[:tile + 1] == [1] * (tile + 1)


def grid(kind, shapes, extra=()):
    out = []
    for dt, D in shapes:
        names = BASE_LAYOUTS + tuple(n for n in POINT_LAYOUTS if n in plan_points(kind, dt, D)) + tuple(extra)
        out += [pytest.param(dt, D, n, id=f"{dt}-D{D}-{n}") for n in names]
    return out


# ------------------------------------------------------------------------------------------------ inputs
class Case:
    """One batch: trees from synth.random_tree, the staged graph and its row_sent=None twin, anchors and distances."""

    def __init__(self, lens, M, seed):
        import ed_gated_gcn_b200 as E
        from ed_gated_gcn_b200 import synth
        rng = np.random.default_rng(seed + 1)
        self.lens = np.asarray(lens, dtype=np.int64)
        self.B, self.N, self.M = len(lens), int(sum(lens)), M
        self.sp = np.concatenate([[0], np.cumsum(self.lens)]).astype(np.int64)
        heads = [synth.random_tree(int(n), rng) for n in lens]
        self.heads = heads
        h = np.concatenate(heads).astype(np.int32) if self.N else np.zeros(0, np.int32)
        self.anchor = (rng.random(self.B) * self.lens).astype(np.int32)
        sp32 = torch.from_numpy(self.sp.astype(np.int32))
        if M > MAX_GRAPH_SENTENCE:
            # the pool of bf16 D = 24 stays staged past build_graph's longest sentence; the pool reads no CSR, so its
            # graph carries sent_ptr and row_sent only, as the span pools of segment.py do
            sp_d = sp32.to(DEV)
            rs = torch.from_numpy(np.repeat(np.arange(self.B), self.lens).astype(np.int32)).to(DEV)
            self.g = E.DepGraph(sp_d, sp_d, sp_d, rs, self.B, self.N, M)
            self.dist = None
        else:
            self.g = E.build_graph(torch.from_numpy(h), sp32, max_len=M, device=DEV)
            # (a batch without rows still passes a valid, unread distance pointer)
            self.dist = E.tree_distance(self.g, torch.from_numpy(self.anchor).to(DEV)) if self.N else \
                torch.zeros(1, dtype=torch.int32, device=DEV)
        self.g_flat = dataclasses.replace(self.g, row_sent=None)
        self.rng = rng

    def graphs(self):
        return (("staged", self.g), ("per_sentence", self.g_flat))

    def rows(self, D, dt, scale=1.0):
        from ed_gated_gcn_b200 import ops
        x = torch.from_numpy(self.rng.standard_normal((max(self.N, 1), D)).astype(np.float32) * scale)[:self.N]
        return ops.as_rows(x.to(DEV), TORCH_DT[dt]) if self.N else ops.alloc_rows(0, D, TORCH_DT[dt], DEV, zero=True)

    def tree_batch(self):
        from ed_gated_gcn_b200 import synth
        return synth.TreeBatch(heads=np.concatenate(self.heads).astype(np.int32) if self.N else np.zeros(0, np.int32),
                               sent_ptr=self.sp.astype(np.int32), anchor=self.anchor, lengths=self.lens.astype(np.int32))


def nan_f32(*shape):
    return torch.full(shape, float("nan"), dtype=torch.float32, device=DEV)


def host(t):
    return t.detach().cpu().double().numpy()


def assert_within(got, want, bound, what):
    got = np.asarray(got, dtype=np.float64)
    err = np.abs(got - want)
    bad = np.argwhere(~(err <= bound))                        # NaN (an unwritten sentinel) fails too
    assert len(bad) == 0, (f"{what}: {len(bad)} of {err.size} off, first {tuple(bad[0])}: got {got[tuple(bad[0])]!r}, "
                           f"want {want[tuple(bad[0])]!r}, bound {bound[tuple(bad[0])]:.3g}")


# ------------------------------------------------------------------------------------------------ C entry points
# Small mirrors of ops.pool_fwd / ops.scores_kl_fwd / ops.head_bwd / ops.aggregate whose outputs start as sentinels.
def rows_ptr(t):
    """L.ptr of a row matrix or of row_sent.  torch reports the data pointer of a 0-row view as NULL; a batch without
    rows passes the address of the view's (never read) allocation instead.  So `h` is not rejected as NULL, and
    `row_sent` reaches the staged launchers, which must send N = 0 to the per-sentence kernels."""
    from ed_gated_gcn_b200 import _lib as L
    p = L.ptr(t)
    return t.untyped_storage().data_ptr() if t is not None and t.numel() == 0 else p


def run_pool(h, g, gates):
    from ed_gated_gcn_b200 import _lib as L, ops
    V, B, D = gates.shape
    pooled, hmax = nan_f32(V, B, D), nan_f32(B, D)
    arg = torch.full((V, B, D), -7, dtype=torch.int32, device=DEV)
    L.call("edg_pool_fwd", rows_ptr(h), L.dt(h), ops.ld(h), L.ptr(g.sent_ptr), B, D, L.ptr(gates), V, L.ptr(pooled),
           L.ptr(arg), rows_ptr(g.row_sent), g.n_rows, g.max_len, L.ptr(hmax), L.stream())
    return pooled, arg, hmax


def run_scores(h, g, gate, v, c, dist, units=True):
    from ed_gated_gcn_b200 import _lib as L, ops
    B, D = gate.shape
    N = h.shape[0]
    scores, kl_b, kl = nan_f32(max(N, 1)), nan_f32(B), nan_f32(1)
    dvu, dcu, uu, sfu = (nan_f32(B, D), nan_f32(B), nan_f32(max(N, 1)), nan_f32(B, D)) if units else (None,) * 4
    L.call("edg_scores_kl_fwd", rows_ptr(h), L.dt(h), ops.ld(h), L.ptr(g.sent_ptr), B, D, L.ptr(gate), L.ptr(v), L.ptr(c),
           L.ptr(dist), ops._dist_flag(dist), L.ptr(scores), L.ptr(kl_b), L.ptr(dvu), L.ptr(dcu),
           L.ptr(uu), L.ptr(sfu), rows_ptr(g.row_sent), g.n_rows, g.max_len, L.stream())
    L.call("edg_sum_scaled", L.ptr(kl_b), B, 1.0 / B, L.ptr(kl), L.stream())
    return scores[:N], kl_b, kl, dvu, dcu, (uu[:N] if units else None), sfu


def run_head_bwd(h, g, gate, v, dist, scores, kl_b, g_kl, g_scores, g_pooled, arg, g_xout, first_pass):
    from ed_gated_gcn_b200 import _lib as L, ops
    B, D = gate.shape
    N = h.shape[0]
    dh = None
    if not first_pass:
        dh = ops.alloc_rows(N, D, h.dtype, DEV)
        dh.as_strided((max(N, 1), ops.ld(dh)), (ops.ld(dh), 1)).fill_(float("nan"))
    dgate = None if first_pass else nan_f32(B, D)
    dv, dc = nan_f32(B, D), nan_f32(B)
    L.call("edg_head_bwd", rows_ptr(h), L.dt(h), ops.ld(h), L.ptr(g.sent_ptr), B, D, L.ptr(gate), L.ptr(v),
           L.ptr(dist), ops._dist_flag(dist), L.ptr(scores), L.ptr(kl_b), L.ptr(g_kl),
           L.ptr(g_scores), L.ptr(g_pooled), L.ptr(arg), rows_ptr(g_xout), ops.ld(g_xout) if g_xout is not None else 0,
           rows_ptr(dh), ops.ld(dh) if dh is not None else 0, L.ptr(dgate), L.ptr(dv), L.ptr(dc), g.max_len,
           rows_ptr(g.row_sent), g.n_rows, L.stream())
    return dh, dgate, dv, dc


def run_aggregate(x, g, mode, out_dtype):
    from ed_gated_gcn_b200 import _lib as L, ops
    N, D = x.shape
    y = ops.alloc_rows(N, D, out_dtype, DEV, min_ld=ops.row_pitch(D, x.dtype))
    y.as_strided((max(N, 1), ops.ld(y)), (ops.ld(y), 1)).fill_(float("nan"))
    L.call("edg_aggregate", rows_ptr(x), L.dt(x), ops.ld(x), rows_ptr(y), L.dt(y), ops.ld(y), N, D, L.ptr(g.row_ptr),
           L.ptr(g.col), mode, L.ptr(g.sent_ptr), rows_ptr(g.row_sent), g.n_graphs, g.max_len, L.stream())
    return y


# ------------------------------------------------------------------------------------------------ softmax bounds
def softmax_rel(x, abs_err=0.0):
    """fp64 softmax of one sentence and a bound on the relative error of its fp32 evaluation.  Inputs off by at most
    abs_err move max-subtracted exponents by 2 abs_err; the subtraction rounds (u |x - m|), expf is within 2 ulp
    (4u), the sum of n terms through a sequential loop and 5 shuffle levels adds (n + 5) u to Z, the division u."""
    m = x.max()
    e = np.exp(x - m)
    num = 2 * abs_err + U * (np.abs(x - m).max() + 4)
    return e / e.sum(), 2 * num + (len(x) + 6) * U


# ------------------------------------------------------------------------------------------------ the pool
POOL_SHAPES = [("bf16", 300), ("f32", 300), ("bf16", 768), ("f32", 768), ("bf16", 64), ("f32", 64), ("bf16", 32),
               ("bf16", 24)]
VIEWS = (1, 2, 3, 5)       # the staged pool launches pairs of views, the per-sentence pool groups of four


@pytest.mark.parametrize("dt,D,layout", grid("pool", POOL_SHAPES))
def test_pool_both_implementations(dt, D, layout):
    seed = D + 7 * len(layout)
    lens, M, _ = make_layout("pool", dt, D, layout, seed)
    case = Case(lens, M, seed)
    V = VIEWS[(BASE_LAYOUTS + POINT_LAYOUTS).index(layout) % 4]
    B, N, sp = case.B, case.N, case.sp
    x = case.rng.standard_normal((N, D)).astype(np.float32)
    x[:, 5 % D] = -np.abs(x[:, 5 % D]) - 0.25                 # a column that is negative everywhere
    live = np.nonzero(case.lens > 1)[0]
    for s in live[::3]:                                       # ties: a sentence of identical rows ...
        x[sp[s]:sp[s + 1]] = x[sp[s]]
    for s in live[1::3]:                                      # ... and a repeated row
        x[sp[s] + 1] = x[sp[s]]
    from ed_gated_gcn_b200 import ops
    h = ops.as_rows(torch.from_numpy(x).to(DEV), TORCH_DT[dt]) if N else case.rows(D, dt)
    gates = (case.rng.random((V, B, D)) + 0.05).astype(np.float32)
    gates[:, ::2, 3 % D] = 0.0                                # gates of exactly 0
    gates[0, 1::2, :] *= 1e-3
    res = {name: run_pool(h, g, torch.from_numpy(gates).to(DEV)) for name, g in case.graphs()}
    # host reference: max_t fl(h_t) * g in fp32 (gates are positive or 0 and rounding is monotone), arg = the first
    # row of the column maximum (the row start where the gate is 0), empty sentences 0 / -1 / 0
    hs = h.float().cpu().numpy()
    want_p = np.zeros((V, B, D), np.float32)
    want_a = np.full((V, B, D), -1, np.int64)
    want_h = np.zeros((B, D), np.float32)
    for s in range(B):
        lo, hi = sp[s], sp[s + 1]
        if hi == lo:
            continue
        m = hs[lo:hi].max(0)
        first = lo + np.argmax(hs[lo:hi] == m, axis=0)
        want_h[s] = m
        want_p[:, s] = m[None, :] * gates[:, s]
        want_a[:, s] = np.where(gates[:, s] != 0, first[None, :], lo)
        prod = hs[lo:hi][None] * gates[:, s][:, None]         # the reference's own maximum of the products
        assert np.array_equal(want_p[:, s], prod.max(1))
    for name, (pooled, arg, hmax) in res.items():
        assert np.array_equal(pooled.cpu().numpy().view(np.int32), want_p.view(np.int32)), f"{name}: pooled"
        assert np.array_equal(arg.cpu().numpy().astype(np.int64), want_a), f"{name}: arg"
        assert np.array_equal(hmax.cpu().numpy().view(np.int32), want_h.view(np.int32)), f"{name}: hmax"


# ------------------------------------------------------------------------------------------------ scores and kl
SCORES_SHAPES = [("bf16", 300), ("f32", 300), ("bf16", 768), ("f32", 768), ("bf16", 64), ("f32", 64), ("bf16", 256),
                 ("bf16", 264), ("bf16", 512), ("bf16", 520), ("bf16", 776), ("bf16", 1024)]


def scores_reference(case, hs, gate, v, c, dist, D_pad):
    """fp64 formulas of edg_scores_kl_fwd on the stored inputs, and element-wise bounds.

    scores_t = sum_d h g v + c.  The kernels round w = g v once, then sum D fp32 products: the staged kernel in four
    accumulators of D_pad / 4 products each, then two additions and + c; the per-sentence kernel per lane (at most
    D_pad / 4 products here) and five shuffle levels.  With depth D_pad / 4 + 8 the bound c_s u sum_d |h g v| holds for
    both; it is 2 - 4 % of the sum of |terms| of one 16-byte chunk (8 bf16 or 4 fp32 products) even at D = 1024, so a
    chunk or a row left out fails.  The other outputs carry the score bound through the softmax (softmax_rel) and
    add the depth of their own sums: kl_b = sum_t P Q, u_t = P (Q - kl) / B, dc = sum_t u, sf = sum_t u_t h_t
    (one fma per row, n deep), dv = sf g."""
    B, D = gate.shape
    cs = D_pad // 4 + 8
    N = hs.shape[0]
    out = {k: np.zeros(s) for k, s in (("scores", N), ("kl_b", B), ("u", N), ("dc", B), ("sf", (B, D)), ("dv", (B, D)))}
    bnd = {k: np.zeros_like(a) for k, a in out.items()}
    for s in range(B):
        lo, hi = case.sp[s], case.sp[s + 1]
        n = hi - lo
        if n == 0:
            continue
        terms = hs[lo:hi] * (gate[s] * v[s])[None]
        sc = terms.sum(1) + c[s]
        es = cs * U * (np.abs(terms).sum(1) + abs(c[s]))
        P, rp = softmax_rel(sc, es.max())
        Q, rq = softmax_rel(dist[lo:hi].astype(np.float64))
        kl = (P * Q).sum()
        ekl = (rp + rq + (n + 9) * U) * kl
        u = P * (Q - kl) / B
        eu = (P * (np.abs(Q - kl) * (rp + 4 * U) + Q * rq + ekl)) / B
        sf = u @ hs[lo:hi]
        esf = eu @ np.abs(hs[lo:hi]) + (n + 2) * U * (np.abs(u) @ np.abs(hs[lo:hi]))
        out["scores"][lo:hi], bnd["scores"][lo:hi] = sc, es
        out["kl_b"][s], bnd["kl_b"][s] = kl, ekl
        out["u"][lo:hi], bnd["u"][lo:hi] = u, eu
        out["dc"][s], bnd["dc"][s] = u.sum(), eu.sum() + (n + 5) * U * np.abs(u).sum()
        out["sf"][s], bnd["sf"][s] = sf, esf
        out["dv"][s], bnd["dv"][s] = sf * gate[s], esf * gate[s] + U * np.abs(sf * gate[s])
    return out, bnd


def _scores_inputs(case, dt, D):
    B = case.B
    h = case.rows(D, dt)
    gate = case.rng.random((B, D)).astype(np.float32)
    v = (case.rng.standard_normal((B, D)) * 0.1).astype(np.float32)
    c = case.rng.standard_normal(B).astype(np.float32)
    return h, gate, v, c


@pytest.mark.parametrize("dt,D,layout", grid("scores", SCORES_SHAPES, SCORES_LAYOUTS))
def test_scores_kl_both_implementations(dt, D, layout):
    seed = 3 * D + 11 * len(layout)
    lens, M, _ = make_layout("scores", dt, D, layout, seed)
    case = Case(lens, M, seed)
    h, gate, v, c = _scores_inputs(case, dt, D)
    dist = case.dist.long() if seed % 2 else case.dist        # int32 and int64 distances
    dev = [torch.from_numpy(a).to(DEV) for a in (gate, v, c)]
    E = 16 // ESIZE[dt]
    want, bnd = scores_reference(case, host(h), gate.astype(np.float64), v.astype(np.float64), c.astype(np.float64),
                                 host(dist), -(-D // E) * E)
    B = case.B
    got = {}
    for name, g in case.graphs():
        scores, kl_b, kl, dvu, dcu, uu, sfu = run_scores(h, g, *dev, dist)
        got[name] = {"scores": host(scores), "kl_b": host(kl_b), "u": host(uu), "dc": host(dcu), "sf": host(sfu),
                     "dv": host(dvu)}
        for k in got[name]:
            assert_within(got[name][k], want[k], bnd[k], f"{name}: {k}")
        # kl = mean(kl_b), summed in fp64 and rounded once
        assert_within(host(kl), np.array([want["kl_b"].mean()]), np.array([bnd["kl_b"].mean() + 2 * U * want["kl_b"].mean()]),
                      f"{name}: kl")
        # without the unit outputs (the kernels skip their last phase): the same scores and kl_b
        s2, k2, _, _, _, _, _ = run_scores(h, g, *dev, dist, units=False)
        assert torch.equal(s2, scores) and torch.equal(k2, kl_b), name
    # the two implementations agree within the sum of their bounds
    for k in bnd:
        assert_within(got["staged"][k], got["per_sentence"][k], 2 * bnd[k], f"staged vs per-sentence: {k}")


def test_scores_rejects_more_than_128_bf16_chunks():
    case = Case([5, 0, 7], 7, 0)
    h, gate, v, c = _scores_inputs(case, "bf16", 1032)
    from ed_gated_gcn_b200 import _lib as L
    for name, g in case.graphs():
        with pytest.raises(L.EdgError, match="status"):
            run_scores(h, g, *(torch.from_numpy(a).to(DEV) for a in (gate, v, c)), case.dist)


# ------------------------------------------------------------------------------------------------ head backward
HEAD_SHAPES = POOL_SHAPES       # bf16 D = 32: exactly one warp per staged block; D = 24: less than one (per-sentence)

# (g_kl, g_scores, g_pooled, g_xout, first pass: dh = dgate = NULL)
HEAD_COMBOS = [(a, b, p, x, False) for a in (0, 1) for b in (0, 1) for p in (0, 1) for x in (0, 1)] + \
              [(1, 1, 0, 0, True), (0, 1, 0, 0, True), (1, 0, 1, 0, True)]


def head_reference(case, hs, gate, v, dist, scores, klb, gk, gs, gp, arg, gx):
    """fp64 formulas of edg_head_bwd (include/edgcn.h) and element-wise bounds.  ds_t = g_kl / B P_t (Q_t - kl_b) +
    g_scores_t from the GIVEN scores and kl_b (softmax_rel with exact inputs); dh = g (ds v + [t == arg] gp + gx) is
    a few fp32 operations on ds (4u); dv = sum_t ds h g, dgate = sum_t h (ds v + gx) + gp h[arg] and dc = sum_t ds are
    sums of n rows (n + 5 deep)."""
    B, D = gate.shape
    N = hs.shape[0]
    out = {"dh": np.zeros((N, D)), "dgate": np.zeros((B, D)), "dv": np.zeros((B, D)), "dc": np.zeros(B)}
    bnd = {k: np.zeros_like(a) for k, a in out.items()}
    g_kl = gk if gk is not None else 0.0
    for s in range(B):
        lo, hi = case.sp[s], case.sp[s + 1]
        n = hi - lo
        if n == 0:
            continue
        H = hs[lo:hi]
        ds, eds = np.zeros(n), np.zeros(n)
        if gk is not None:
            P, rp = softmax_rel(scores[lo:hi])
            Q, rq = softmax_rel(dist[lo:hi].astype(np.float64))
            t = g_kl / B * P * (Q - klb[s])
            ds += t
            eds += abs(g_kl) / B * P * (np.abs(Q - klb[s]) * (rp + 4 * U) + Q * rq) + 4 * U * np.abs(t)
        if gs is not None:
            ds += gs[lo:hi]
            eds += 2 * U * np.abs(gs[lo:hi])
        onarg = (arg[s][None, :] == np.arange(lo, hi)[:, None]) if gp is not None else np.zeros((n, D), bool)
        gpv = gp[s] if gp is not None else np.zeros(D)
        gxv = gx[lo:hi] if gx is not None else np.zeros((n, D))
        coef = ds[:, None] * v[s][None] + onarg * gpv[None] + gxv
        acoef = np.abs(ds[:, None] * v[s][None]) + onarg * np.abs(gpv[None]) + np.abs(gxv)
        out["dh"][lo:hi] = gate[s][None] * coef
        bnd["dh"][lo:hi] = gate[s][None] * (eds[:, None] * np.abs(v[s][None]) + 4 * U * acoef)
        out["dgate"][s] = (H * coef).sum(0)
        bnd["dgate"][s] = (eds @ np.abs(H)) * np.abs(v[s]) + (n + 5) * U * (np.abs(H) * acoef).sum(0)
        out["dv"][s] = (ds @ H) * gate[s]
        bnd["dv"][s] = (eds @ np.abs(H) + (n + 5) * U * (np.abs(ds) @ np.abs(H))) * gate[s]
        out["dc"][s] = ds.sum()
        bnd["dc"][s] = eds.sum() + (n + 5) * U * np.abs(ds).sum()
    return out, bnd


@pytest.mark.parametrize("dt,D,layout", grid("head", HEAD_SHAPES))
def test_head_bwd_both_implementations(dt, D, layout):
    seed = 5 * D + 13 * len(layout)
    lens, M, _ = make_layout("head", dt, D, layout, seed)
    case = Case(lens, M, seed)
    B, N, rng = case.B, case.N, case.rng
    h = case.rows(D, dt)
    hs = host(h)
    gate = rng.random((B, D)).astype(np.float32)
    v = (rng.standard_normal((B, D)) * 0.1).astype(np.float32)
    scores = (rng.standard_normal(max(N, 1)) * 2).astype(np.float32)[:N]
    klb = rng.random(B).astype(np.float32)
    gs = rng.standard_normal(max(N, 1)).astype(np.float32)[:N]
    gp = rng.standard_normal((B, D)).astype(np.float32)
    # arg-max rows built on the host: a row of the sentence, -1 for some columns and for every empty sentence
    arg = np.full((B, D), -1, np.int32)
    for s in range(B):
        if case.lens[s]:
            arg[s] = case.sp[s] + rng.integers(0, case.lens[s], D)
            arg[s, rng.random(D) < 0.2] = -1
    gx_t = case.rows(D, dt, scale=0.5)
    gx = host(gx_t)
    dist = case.dist.long() if seed % 2 else case.dist
    gk = np.float32(0.7)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(DEV)
    dev_in = dict(gate=t(gate), v=t(v), scores=t(scores) if N else nan_f32(1), kl_b=t(klb))
    dh_u = U_BF16 if dt == "bf16" else 0.0
    for kl_on, sc_on, p_on, x_on, first in HEAD_COMBOS:
        want, bnd = head_reference(case, hs, gate.astype(np.float64), v.astype(np.float64), host(dist),
                                   scores.astype(np.float64), klb.astype(np.float64), float(gk) if kl_on else None,
                                   gs.astype(np.float64) if sc_on else None, gp.astype(np.float64) if p_on else None,
                                   arg, gx if x_on else None)
        bnd["dh"] = bnd["dh"] + dh_u * (np.abs(want["dh"]) + bnd["dh"])     # the store rounds once to bf16
        got = {}
        what = f"g_kl={kl_on} g_scores={sc_on} g_pooled={p_on} g_xout={x_on} first_pass={first}"
        for name, g in case.graphs():
            dh, dgate, dv, dc = run_head_bwd(
                h, g, dev_in["gate"], dev_in["v"], dist, dev_in["scores"], dev_in["kl_b"],
                torch.tensor([float(gk)], dtype=torch.float32, device=DEV) if kl_on else None, t(gs) if sc_on and N else (nan_f32(1) if sc_on else None),
                t(gp) if p_on else None, t(arg) if p_on else None, gx_t if x_on else None, first)
            got[name] = {"dv": host(dv), "dc": host(dc)}
            if not first:
                got[name]["dh"], got[name]["dgate"] = host(dh), host(dgate)
            for k in got[name]:
                assert_within(got[name][k], want[k], bnd[k], f"{name} {what}: {k}")
        for k in got["staged"]:
            assert_within(got["staged"][k], got["per_sentence"][k], 2 * bnd[k], f"staged vs per-sentence {what}: {k}")


# ------------------------------------------------------------------------------------------------ aggregation
AGG_SHAPES = [("bf16", 300), ("f32", 300), ("bf16", 64)]


@pytest.mark.parametrize("dt,D,layout", [pytest.param(dt, D, n, id=f"{dt}-D{D}-{n}") for dt, D in AGG_SHAPES
                                         for n in BASE_LAYOUTS])
def test_aggregate_staged_and_flat(dt, D, layout):
    """edg_aggregate modes 0 and 1 on the staged graph and on the row_sent=None graph (the flat kernel), fp32 / bf16 /
    mixed output, against the fp64 adjacency product (gcn.py:35, 41) and each other."""
    seed = 17 * D + len(layout)
    lens, M, _ = make_layout("pool", dt, D, layout, seed)
    case = Case(lens, M, seed)
    if case.N == 0:
        for name, g in case.graphs():
            y = run_aggregate(case.rows(D, dt), g, 0, TORCH_DT[dt])
            assert y.shape == (0, D), name
        return
    x = case.rows(D, dt)
    xs = host(x)
    ah = adj_hat(case.tree_batch())
    K = int(np.diff(case.g.row_ptr.cpu().numpy()).max())      # the longest CSR row: the depth of every fp32 sum
    wants = {0: (ah @ xs, abs(ah) @ np.abs(xs)), 1: (ah.T @ xs, abs(ah.T) @ np.abs(xs))}
    for mode, (want, mag) in wants.items():
        for out_dt in ("f32", "bf16"):
            ys = {}
            for name, g in case.graphs():
                y = run_aggregate(x, g, mode, TORCH_DT[out_dt])
                assert_rows_close(y.float(), want, mag, f"{name} mode {mode} {dt}->{out_dt}")
                if dt == out_dt == "f32":                     # K + 2 roundings of fp32 sums, products and the scale
                    assert_within(host(y), want, (K + 2) * U * (mag + np.abs(want)), f"{name} mode {mode} f32")
                ys[name] = host(y)
            # the two implementations are each within one bar of the fp64 product
            bar = 2 * 8e-3 * (mag + np.abs(want)) if "bf16" in (dt, out_dt) else 2 * (K + 2) * U * (mag + np.abs(want))
            assert_within(ys["staged"], ys["per_sentence"], bar, f"staged vs flat mode {mode} {dt}->{out_dt}")
