"""The trigger-pair kernels of csrc/edg_pairs.cu one by one, through the C ABI, against fp64 restatements of their
formulas (include/edgcn.h, "Trigger pairs") with element-wise bounds.

Each pair p reads its own copy of its sentence's rows, so every reference is built on the expanded batch (the
sentence of every pair copied once, pair p's rows starting at pair_row_ptr[p], test_gpu_j._expand): the scores /
kl and head-backward formulas are the per-sentence ones of test_gpu_i with B = P, and d h of a sentence row is the
sum over the sentence's pairs of what each copy of the row receives.  Under gate dropout the rows a pair reads are
rebuilt bit for bit (T(h * scale) where the pair's mask keeps an element, 0 where it drops it); under the sigmoid
head z = sigmoid(g_p * h~) is formed in fp64 with a bound of one ulp of T plus a few u.

The grid covers both chunk sizes (8 bf16 / 4 fp32 columns per 16-byte chunk): a single column pass, the start of
the second pass, a partial last chunk, the 128-chunk limit and the rejection just past it; sentences of 1 - 5 rows
(4 rows in flight in the scores kernel, 2 in the pool), 31 - 33 and 63 - 65 rows (lane-strided softmax loops),
anchors in descending, shuffled and repeated order, sentences without pairs at both ends, an empty sentence that
owns pairs, P = 0 with rows present and a batch of empty sentences.  `h` is always a column slice of a wider
allocation whose extra columns hold a large finite value, so a kernel that lets padding into a result fails.

Every output starts as a sentinel (NaN, -7 for `arg`, NaN across the whole `dh` allocation), so an element that no
thread writes fails deterministically; the outputs that only the C ABI reaches (u_unit, sf_unit, dv / dc next to dh)
are requested.  The fp64 backward formulas are checked once against torch.autograd on the CPU."""
import types

import numpy as np
import pytest
import torch

from gpu_util import DEV
from test_gpu_c_models import _dropout_mask_numpy
from test_gpu_i_staged_windows import (U, U_BF16, assert_within, head_reference, host, nan_f32, rows_ptr,
                                       scores_reference, softmax_rel)
from test_gpu_j_pairs import _expand, _layout, _lengths_batch

U_T = {"bf16": U_BF16, "f32": U}
TORCH_DT = {"bf16": torch.bfloat16, "f32": torch.float32}
ELEMS = {"bf16": 8, "f32": 4}                 # columns per 16-byte chunk
BIG = 2.0 ** 100                              # what the columns past D of `h` hold: finite, exact in both dtypes
SEED = 0x1234_5678_9ABC_DEF1 >> 1
KEEP_PATTERN = 0.4375                         # d h_1 before edg_views_bwd_drop_pairs adds into it

# ------------------------------------------------------------------------------------------------ the grid
WIDTHS = [("bf16", D) for D in (20, 300, 256, 264, 768, 1024, 1020)] + \
         [("f32", D) for D in (20, 128, 132, 302, 768, 1024)]
LAYOUTS = ("mixed", "long", "512", "short", "lanes", "order", "empty_owner", "no_pairs", "all_empty")
PAST_LIMIT = {"bf16": 1032, "f32": 1028}
KINDS = ("plain", "drop", "sig", "sig_drop")   # edg_*_pairs, edg_*_drop_pairs, edg_*_sig_pairs without / with seed
DROP_P = (0.0, 0.25, 0.9)


def layouts_for(D):
    """Host references stay affordable: the 512-row, 512-pair sentence at D <= 64 only, and layouts of at most about
    20k pair rows ("long" has 12.5k) at D >= 768."""
    return tuple(n for n in LAYOUTS if not (n == "512" and D > 64) and not (n == "long" and D > 302))


def grid(widths=WIDTHS, layouts=None):
    return [pytest.param(dt, D, n, id=f"{dt}-D{D}-{n}") for dt, D in widths for n in (layouts or layouts_for(D))]


def pair_layout(name):
    """(TreeBatch, pair_ptr, anchor): the layouts of test_gpu_j and those of this file."""
    if name in ("mixed", "long", "512"):
        return _layout(name)
    lens, per = {
        # every sentence length the scores kernel's 4 rows in flight and the pool's 2 can leave partial
        "short": ([1, 2, 3, 4, 5, 3, 1], [[0], [1, 0], [2, 0, 1], [3, 3, 0], [4, 1, 2, 0], [1], [0]]),
        # the lane-strided softmax loops: one row short of, exactly and one past one and two warps
        "lanes": ([31, 32, 33, 63, 64, 65], [[0, 30, 15], [31, 0], [32, 1, 16], [62, 0], [63, 31, 5], [64, 0, 32]]),
        # no pairs in the first and last sentences, descending, shuffled and repeated anchors
        "order": ([6, 9, 4, 7, 5, 8], [[], [8, 5, 3, 1, 0], [2, 0, 3, 1, 1, 3], [6, 6, 6], [0, 4, 2], []]),
        # an empty sentence that owns pairs (its anchors index nothing): their copies have no rows
        "empty_owner": ([4, 0, 5, 0], [[1], [0, 0], [2, 4], [0]]),
        # rows but no pairs: the head backward writes d h = 0 and nothing else
        "no_pairs": ([5, 3, 7], [[], [], []]),
        # every sentence empty, two of them with pairs
        "all_empty": ([0, 0, 0], [[0], [], [0, 0]]),
    }[name]
    b = _lengths_batch(lens, seed=len(name))
    pp = np.zeros(len(per) + 1, dtype=np.int32)
    pp[1:] = np.cumsum([len(p) for p in per])
    return b, pp, np.asarray([a for p in per for a in p], dtype=np.int32)


class PairCase:
    """One batch of pairs on the host (sentence rows, the expanded batch) and, on demand, on the device."""

    def __init__(self, name, seed):
        b, pp, an = pair_layout(name)
        self.sp = b.sent_ptr.astype(np.int64)
        self.S, self.N = len(self.sp) - 1, int(self.sp[-1])
        self.pp = pp.astype(np.int64)
        self.P = int(self.pp[-1])
        self.pair_sent = np.repeat(np.arange(self.S), np.diff(self.pp))
        self.anchor = an.astype(np.int64)
        eb, rows = _expand(b, pp, an)
        self.prp = eb.sent_ptr.astype(np.int64)              # pair_row_ptr
        self.R = int(self.prp[-1])
        self.rows = rows.numpy().astype(np.int64)            # expanded row -> sentence row
        self.row_pair = np.repeat(np.arange(self.P), np.diff(self.prp))
        self.row_sent = np.repeat(np.arange(self.S), np.diff(self.sp))
        self.npairs_of_row = np.diff(self.pp)[self.row_sent]  # depth of every sum over a row's pairs
        self.exp = types.SimpleNamespace(sp=self.prp)        # the expanded batch as test_gpu_i's references see it
        self.rng = np.random.default_rng(seed)
        self._dev = None

    @property
    def dev(self):
        if self._dev is None:
            self._dev = types.SimpleNamespace(
                sent_ptr=i32(self.sp), row_sent=i32(self.row_sent), pair_ptr=i32(self.pp), pair_sent=i32(self.pair_sent),
                pair_row_ptr=i32(self.prp), pair_start=i32(self.sp[self.pair_sent]), anchor=i32(self.anchor))
        return self._dev

    def expanded_arg(self, arg, per_pair):
        """Sentence rows of `arg` ([P,D] per pair, or [S,D] per sentence) -> rows of each pair's copy, -1 outside."""
        a = arg if per_pair else arg[self.pair_sent]
        beg = self.sp[self.pair_sent][:, None]
        n = np.diff(self.sp)[self.pair_sent][:, None]
        loc = a.astype(np.int64) - beg
        return np.where((loc >= 0) & (loc < n), self.prp[:-1, None] + loc, -1)

    def sum_to_rows(self, a):
        """Sum per-pair row values [R,...] into the sentence rows [N,...] (fp64)."""
        out = np.zeros((self.N,) + a.shape[1:])
        np.add.at(out, self.rows, a)
        return out


def _on_device(a, dtype):
    """A device copy of `a`; an empty one keeps a one-element allocation so rows_ptr passes a non-NULL address."""
    t = torch.zeros(max(a.size, 1), dtype=dtype, device=DEV)
    if a.size:
        t[:a.size] = torch.from_numpy(np.ascontiguousarray(a).reshape(-1)).to(DEV)
    return t[:a.size].view(a.shape)


def i32(a):
    return _on_device(np.asarray(a, dtype=np.int32), torch.int32)


def f32(a):
    return _on_device(np.asarray(a, dtype=np.float32), torch.float32)


def to_T(a, dt):
    """fp32 values rounded to T (round to nearest even, as __float2bfloat16_rn)."""
    a = np.asarray(a, dtype=np.float32)
    return a if dt == "f32" else torch.from_numpy(a).to(torch.bfloat16).float().numpy()


def wide_rows(x32, dt):
    """x as rows of T in a column slice of a wider allocation: one extra 16-byte chunk per row, every column past D
    (the pitch padding of the last chunk too) holding BIG."""
    N, D = x32.shape
    E = ELEMS[dt]
    ld = -(-D // E) * E + E
    base = torch.full((max(N, 1), ld), BIG, dtype=TORCH_DT[dt], device=DEV)
    base[:N, :D] = torch.from_numpy(x32).to(DEV).to(TORCH_DT[dt])
    return base[:N, :D]


def nan_rows(N, D, dt):
    """A d h row matrix at the default pitch, NaN across the whole allocation (padding columns included)."""
    from ed_gated_gcn_b200 import ops
    dh = ops.alloc_rows(N, D, TORCH_DT[dt], DEV)
    full(dh).fill_(float("nan"))
    return dh


def full(rows):
    """The whole allocation behind a row matrix, padding columns included."""
    return rows.as_strided((max(rows.shape[0], 1), rows.stride(0)), (rows.stride(0), 1))


def drop_masks(pc, stream_id, p, D):
    """keep / (1 - p) of every (pair row, column) under dropout stream `stream_id` [R,D] fp32."""
    return _dropout_mask_numpy(SEED, stream_id, float(np.float32(p)), pc.R, D)


def masked_rows(hs32, pc, M, dt):
    """The rows each pair reads [R,D] fp32: T(h * scale) where kept, +0 where dropped (M = None: the rows as stored)."""
    x = hs32[pc.rows]
    if M is None:
        return x
    return np.where(M > 0, to_T(x * M, dt), np.float32(0.0)).astype(np.float32)


# ------------------------------------------------------------------------------------------------ C entry points
# Mirrors of ops.scores_kl_*pairs_fwd / head_bwd_*pairs / pool_drop_pairs / views_bwd_*pairs /
# trigger_scatter_add_pairs whose outputs start as sentinels.
def _L():
    from ed_gated_gcn_b200 import _lib as L, ops
    return L, ops


def _masked(kind):
    return kind in ("drop", "sig_drop")


def run_scores(kind, pc, h, gate, v, c, dist, stream_id=0, p=0.0, units=True, seed=None, keep=None):
    """`keep`: a dict that receives the output tensors before the call (to check them after a refused call)."""
    L, ops = _L()
    P, D, R = pc.P, h.shape[1], pc.R
    d = pc.dev
    out = {"scores": nan_f32(max(R, 1)), "kl_b": nan_f32(max(P, 1))}
    if units:
        out.update(dv=nan_f32(max(P, 1), D), dc=nan_f32(max(P, 1)))
        if kind in ("plain", "drop"):                     # the outputs ops.py never requests
            out.update(u=nan_f32(max(R, 1)), sf=nan_f32(max(P, 1), D))
    if keep is not None:
        keep.update(out)
    o = {k: L.ptr(out.get(k)) for k in ("scores", "kl_b", "dv", "dc", "u", "sf")}
    args = [rows_ptr(h), L.dt(h), ops.ld(h), rows_ptr(d.sent_ptr), rows_ptr(d.pair_sent), rows_ptr(d.pair_row_ptr), P, D,
            rows_ptr(gate), rows_ptr(v), L.ptr(c), rows_ptr(dist), ops._dist_flag(dist), o["scores"], o["kl_b"], o["dv"],
            o["dc"]]
    seed = seed if seed is not None else torch.tensor([SEED], dtype=torch.int64, device=DEV)
    if kind == "plain":
        L.call("edg_scores_kl_pairs_fwd", *args, o["u"], o["sf"], L.stream())
    elif kind == "drop":
        L.call("edg_scores_kl_drop_pairs_fwd", *args, o["u"], o["sf"], L.ptr(seed), stream_id, float(p), L.stream())
    else:
        L.call("edg_scores_kl_sig_pairs_fwd", *args, L.ptr(seed) if kind == "sig_drop" else None, stream_id, float(p),
               L.stream())
    return {k: (t[:R] if k in ("scores", "u") else t[:P]) for k, t in out.items()}


def run_head(kind, pc, h, gate, v, dist, scores, kl_b, g_kl, g_scores, g_pooled, arg, mmax, full_pass, stream_id=0,
             p=0.0, seed=None, keep=None):
    """The first pass (dv, dc) or the full pass (dh, dgate and dv, dc next to them)."""
    L, ops = _L()
    P, D, N, R = pc.P, h.shape[1], pc.N, pc.R
    d = pc.dev
    dt = "bf16" if h.dtype == torch.bfloat16 else "f32"
    dh = nan_rows(N, D, dt) if full_pass else None
    dgate = nan_f32(max(P, 1), D) if full_pass else None
    dv, dc, ds_ws = nan_f32(max(P, 1), D), nan_f32(max(P, 1)), nan_f32(max(R, 1))
    if keep is not None:
        keep.update(dv=dv, dc=dc, ds_ws=ds_ws, **({"dh": full(dh), "dgate": dgate} if full_pass else {}))
    args = [rows_ptr(h), L.dt(h), ops.ld(h), rows_ptr(d.sent_ptr), pc.S, rows_ptr(d.row_sent) if N else None, N,
            rows_ptr(d.pair_ptr), rows_ptr(d.pair_sent), rows_ptr(d.pair_row_ptr), P, D, rows_ptr(gate), rows_ptr(v),
            rows_ptr(dist), ops._dist_flag(dist), rows_ptr(scores), rows_ptr(kl_b), L.ptr(g_kl), rows_ptr(g_scores),
            rows_ptr(g_pooled), rows_ptr(arg)]
    outs = [rows_ptr(dh), ops.ld(dh) if dh is not None else 0, L.ptr(dgate), L.ptr(dv), L.ptr(dc), L.ptr(ds_ws)]
    seed = seed if seed is not None else torch.tensor([SEED], dtype=torch.int64, device=DEV)
    if kind == "plain":
        L.call("edg_head_bwd_pairs", *args, *outs, L.stream())
    else:
        name = "edg_head_bwd_drop_pairs" if kind == "drop" else "edg_head_bwd_sig_pairs"
        L.call(name, *args, rows_ptr(mmax), *outs, L.ptr(seed) if _masked(kind) else None, stream_id, float(p), L.stream())
    return {"dh": dh, "dgate": dgate[:P] if full_pass else None, "dv": dv[:P], "dc": dc[:P], "ds_ws": ds_ws}


def run_pool(pc, h, gates, stream0, p):
    L, ops = _L()
    V, P, D = gates.shape
    d = pc.dev
    pooled, mmax = nan_f32(V, max(P, 1), D), nan_f32(V, max(P, 1), D)
    arg = torch.full((V, max(P, 1), D), -7, dtype=torch.int32, device=DEV)
    seed = torch.tensor([SEED], dtype=torch.int64, device=DEV)
    L.call("edg_pool_drop_pairs", rows_ptr(h), L.dt(h), ops.ld(h), rows_ptr(d.sent_ptr), rows_ptr(d.pair_sent),
           rows_ptr(d.pair_row_ptr), P, D, rows_ptr(gates), V, L.ptr(seed), stream0, float(p), L.ptr(pooled), L.ptr(arg),
           L.ptr(mmax), L.stream())
    return pooled[:, :P], arg[:, :P], mmax[:, :P]


# ------------------------------------------------------------------------------------------------ fp64 references
def sig_values(X, gate, dt):
    """z = sigmoid(g_p * h~) [R,D] in fp64 and a bound on the kernels' T(sigmoid) of the fp32 product: one ulp of T,
    a few u of expf / add / divide, and the rounding of g h moved through the slope z (1 - z)."""
    gh = gate * X
    z = 1.0 / (1.0 + np.exp(-gh))
    return z, (2 * U_T[dt] + 8 * U) * z + U * np.abs(gh) * z * (1 - z)


def pair_scores_ref(pc, X, gate, v, c, dist, D_pad, sig=False, dt="f32"):
    """edg_scores_kl_*pairs_fwd on the rows the pairs read (X [R,D]): scores, kl_b, u, dc, sf, dv.  Without the
    sigmoid these are test_gpu_i's per-sentence formulas on the expanded batch with B = P.  With it the rows are
    z = sigmoid(g h~) against v (unit gate): the bounds of scores_reference plus what the error of z adds."""
    if not sig:
        return scores_reference(pc.exp, X, gate, v, c, dist, D_pad)
    z, ez = sig_values(X, gate[pc.row_pair], dt)
    P, D = gate.shape
    cs = D_pad // 4 + 8
    out = {k: np.zeros(s) for k, s in (("scores", pc.R), ("kl_b", P), ("dc", P), ("dv", (P, D)))}
    bnd = {k: np.zeros_like(a) for k, a in out.items()}
    for p in range(P):
        lo, hi = pc.prp[p], pc.prp[p + 1]
        n = hi - lo
        if n == 0:
            continue
        Z, EZ = z[lo:hi], ez[lo:hi]
        terms = Z * v[p][None]
        sc = terms.sum(1) + c[p]
        es = cs * U * (np.abs(terms).sum(1) + abs(c[p])) + EZ @ np.abs(v[p])
        Pt, rp = softmax_rel(sc, es.max())
        Qt, rq = softmax_rel(dist[lo:hi].astype(np.float64))
        kl = (Pt * Qt).sum()
        ekl = (rp + rq + (n + 9) * U) * kl
        u = Pt * (Qt - kl) / P
        eu = (Pt * (np.abs(Qt - kl) * (rp + 4 * U) + Qt * rq + ekl)) / P
        out["scores"][lo:hi], bnd["scores"][lo:hi] = sc, es
        out["kl_b"][p], bnd["kl_b"][p] = kl, ekl
        out["dc"][p], bnd["dc"][p] = u.sum(), eu.sum() + (n + 5) * U * np.abs(u).sum()
        out["dv"][p] = u @ Z
        bnd["dv"][p] = eu @ Z + np.abs(u) @ EZ + (n + 2) * U * (np.abs(u) @ Z)
    return out, bnd


def pair_head_ref(pc, X, M, gate, v, dist, scores, klb, gk, gs, gp, arg_x, sig=False, dt="f32"):
    """edg_head_bwd_*pairs on the rows the pairs read (X [R,D]) and their masks (M [R,D] = keep / (1 - p), None
    without dropout): dgate, dv, dc per pair, and dh of the sentence rows = the fp64 sum over the row's pairs of what
    each copy receives, M * (ds g v [z (1 - z)] + [t = arg_p] g g_pooled).  `arg_x` [P,D] are the arg-max rows in the
    expanded batch (-1: none).  The bound on dh is the sum of the per-pair bounds plus the depth of the pair loop."""
    P, D = gate.shape
    if not sig:
        out, bnd = head_reference(pc.exp, X, gate, v, dist, scores, klb, gk, gs, gp, arg_x, None)
        dh_x, edh_x = out.pop("dh"), bnd.pop("dh")
        GP = np.abs(gp[pc.row_pair]) if gp is not None else 0.0
        mag_x = gate[pc.row_pair] * (np.abs(_ds_only(pc, gate, dist, scores, klb, gk, gs)[0])[:, None]
                                     * np.abs(v[pc.row_pair]) + _onarg(pc, arg_x, D) * GP)
    else:
        z, ez = sig_values(X, gate[pc.row_pair], dt)
        sl = z * (1 - z)
        esl = ez * np.abs(1 - 2 * z) + ez ** 2 + 2 * U * sl
        ds, eds = _ds_only(pc, gate, dist, scores, klb, gk, gs)
        on = _onarg(pc, arg_x, D)
        G, Vv = gate[pc.row_pair], v[pc.row_pair]
        GP = gp[pc.row_pair] if gp is not None else np.zeros_like(G)
        t_ds = ds[:, None] * G * Vv * sl
        dh_x = t_ds + on * G * GP
        mag_x = np.abs(t_ds) + on * np.abs(G * GP)
        edh_x = np.abs(G * Vv) * (eds[:, None] * sl + np.abs(ds)[:, None] * esl) + 4 * U * mag_x
        out = {"dgate": np.zeros((P, D)), "dv": np.zeros((P, D)), "dc": np.zeros(P)}
        bnd = {k: np.zeros_like(a) for k, a in out.items()}
        Y, eY = sl * X, esl * np.abs(X) + 2 * U * np.abs(sl * X)
        for p in range(P):
            lo, hi = pc.prp[p], pc.prp[p + 1]
            n = hi - lo
            if n == 0:
                continue
            a_ds, a_eds = ds[lo:hi], eds[lo:hi]
            out["dv"][p] = a_ds @ z[lo:hi]
            bnd["dv"][p] = a_eds @ z[lo:hi] + np.abs(a_ds) @ ez[lo:hi] + (n + 5) * U * (np.abs(a_ds) @ z[lo:hi])
            sg = a_ds @ Y[lo:hi]
            esg = a_eds @ np.abs(Y[lo:hi]) + np.abs(a_ds) @ eY[lo:hi] + (n + 5) * U * (np.abs(a_ds) @ np.abs(Y[lo:hi]))
            pool = np.zeros(D)
            if gp is not None:
                ok = arg_x[p] >= 0
                pool[ok] = gp[p][ok] * X[arg_x[p][ok], np.nonzero(ok)[0]]
            out["dgate"][p] = v[p] * sg + pool
            bnd["dgate"][p] = np.abs(v[p]) * esg + 2 * U * (np.abs(v[p] * sg) + np.abs(pool))
            out["dc"][p] = a_ds.sum()
            bnd["dc"][p] = a_eds.sum() + (n + 5) * U * np.abs(a_ds).sum()
    m = np.ones_like(dh_x) if M is None else M.astype(np.float64)
    depth = (pc.npairs_of_row + 2)[:, None] * U
    out["dh"] = pc.sum_to_rows(m * dh_x)
    bnd["dh"] = pc.sum_to_rows(m * (edh_x + 2 * U * mag_x)) + depth * pc.sum_to_rows(m * mag_x)
    return out, bnd


def _onarg(pc, arg_x, D):
    """[R,D]: the expanded row is its pair's arg-max row of the column."""
    if arg_x is None or pc.R == 0:
        return np.zeros((pc.R, D), dtype=bool)
    return arg_x[pc.row_pair] == np.arange(pc.R)[:, None]


def _ds_only(pc, gate, dist, scores, klb, gk, gs):
    """ds_t = g_kl / P P_t (Q_t - kl_b) + g_scores_t from the given scores and kl_b, and its bound (as head_reference)."""
    P = gate.shape[0]
    ds, eds = np.zeros(pc.R), np.zeros(pc.R)
    for p in range(P):
        lo, hi = pc.prp[p], pc.prp[p + 1]
        if hi == lo:
            continue
        if gk is not None:
            Pt, rp = softmax_rel(scores[lo:hi])
            Qt, rq = softmax_rel(dist[lo:hi].astype(np.float64))
            t = gk / P * Pt * (Qt - klb[p])
            ds[lo:hi] += t
            eds[lo:hi] += abs(gk) / P * Pt * (np.abs(Qt - klb[p]) * (rp + 4 * U) + Qt * rq) + 4 * U * np.abs(t)
        if gs is not None:
            ds[lo:hi] += gs[lo:hi]
            eds[lo:hi] += 2 * U * np.abs(gs[lo:hi])
    return ds, eds


# ------------------------------------------------------------------------------------------------ reference self-check
def _autograd_case(sig, masked):
    """fp64 torch forward of one small batch of pairs and the gradients the references restate."""
    pc = PairCase("order", 3)
    rng = np.random.default_rng(11 + 2 * sig + masked)
    D, P, R = 6, pc.P, pc.R
    hs = rng.standard_normal((pc.N, D))
    M = np.where(rng.random((R, D)) < 0.3, 0.0, 1.25) if masked else None
    gate, v = rng.random((P, D)) + 0.1, rng.standard_normal((P, D))
    c, dist = rng.standard_normal(P), rng.integers(0, 9, R).astype(np.float64)
    gk, gs, gp = 0.7, rng.standard_normal(R), rng.standard_normal((P, D))
    arg_x = np.stack([pc.prp[p] + rng.integers(0, pc.prp[p + 1] - pc.prp[p], D) for p in range(P)])
    arg_x[:, 1] = -1
    th, tg, tv, tc = (torch.tensor(a, requires_grad=True) for a in (hs, gate, v, c))
    X = th[torch.from_numpy(pc.rows)] * (torch.from_numpy(M) if masked else 1.0)
    rp = torch.from_numpy(pc.row_pair)
    sc = ((torch.sigmoid(tg[rp] * X) * tv[rp]) if sig else (X * (tg * tv)[rp])).sum(1) + tc[rp]
    kl_b = []
    for p in range(P):
        lo, hi = int(pc.prp[p]), int(pc.prp[p + 1])
        kl_b.append((torch.softmax(sc[lo:hi], 0) * torch.softmax(torch.from_numpy(dist[lo:hi]), 0)).sum())
    kl = torch.stack(kl_b).mean()
    ok = torch.from_numpy(arg_x >= 0)
    Xa = X[torch.from_numpy(np.maximum(arg_x, 0)), torch.arange(D)[None, :]]
    pooled = torch.where(ok, tg * Xa, torch.zeros(()))
    loss = gk * kl + (torch.from_numpy(gs) * sc).sum() + (torch.from_numpy(gp) * pooled).sum()
    units = torch.autograd.grad(kl, (sc, tv, tc), retain_graph=True)
    grads = torch.autograd.grad(loss, (th, tg, tv, tc))
    return pc, locals()


@pytest.mark.parametrize("sig", [False, True], ids=["linear", "sigmoid"])
@pytest.mark.parametrize("masked", [False, True], ids=["rows", "masked"])
def test_pair_references_match_autograd(sig, masked):
    """The restated backward formulas (d kl / d (scores, v, c) of the scores pass, ds / dgate / dv / dc / dh of the
    head backward, the sum of d h over a sentence's pairs, the mask and the sigmoid slope) against torch.autograd of
    the fp64 forward, so a derivation error cannot hide in a reference the kernels agree with."""
    pc, t = _autograd_case(sig, masked)
    X = (t["X"]).detach().numpy()
    gate, v, c, dist = t["gate"], t["v"], t["c"], t["dist"]
    want_s, _ = pair_scores_ref(pc, X, gate, v, c, dist, 8, sig=sig)
    d_sc, d_v, d_c = (a.numpy() for a in t["units"])
    assert np.allclose(want_s["scores"], t["sc"].detach().numpy(), rtol=1e-12, atol=1e-12)
    assert np.allclose(want_s["kl_b"], torch.stack(t["kl_b"]).detach().numpy(), rtol=1e-12, atol=1e-12)
    if not sig:
        assert np.allclose(want_s["u"], d_sc, rtol=1e-10, atol=1e-13)
        assert np.allclose(want_s["sf"] * gate, d_v, rtol=1e-10, atol=1e-13)
    assert np.allclose(want_s["dv"], d_v, rtol=1e-10, atol=1e-13)
    assert np.allclose(want_s["dc"], d_c, rtol=1e-10, atol=1e-13)
    want, _ = pair_head_ref(pc, X, t["M"], gate, v, dist, want_s["scores"], want_s["kl_b"], t["gk"], t["gs"], t["gp"],
                            t["arg_x"], sig=sig)
    g_h, g_g, g_v, g_c = (a.numpy() for a in t["grads"])
    assert np.allclose(want["dh"], g_h, rtol=1e-10, atol=1e-13)
    assert np.allclose(want["dgate"], g_g, rtol=1e-10, atol=1e-13)
    assert np.allclose(want["dv"], g_v, rtol=1e-10, atol=1e-13)
    assert np.allclose(want["dc"], g_c, rtol=1e-10, atol=1e-13)


# ------------------------------------------------------------------------------------------------ scores and head
def _inputs(pc, dt, D):
    rng = pc.rng
    x = rng.standard_normal((pc.N, D)).astype(np.float32)
    hs32 = to_T(x, dt)
    gate = rng.random((pc.P, D)).astype(np.float32)
    gate[:, 3 % D] = 0.0                                      # gates of exactly 0
    v = (rng.standard_normal((pc.P, D)) * 0.1).astype(np.float32)
    c = rng.standard_normal(pc.P).astype(np.float32)
    dist = rng.integers(0, 9, pc.R).astype(np.int32)
    return x, hs32, gate, v, c, dist


GRAD_SUBSETS = [(k, s, p) for k in (0, 1) for s in (0, 1) for p in (0, 1)]


@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("dt,D,layout", grid())
def test_scores_and_head_pairs(kind, dt, D, layout):
    """edg_scores_kl{,_drop,_sig}_pairs_fwd and edg_head_bwd{,_drop,_sig}_pairs: int32 or int64 distances, c = NULL
    on every other layout, p in {0, 0.25, 0.9} under dropout (at p = 0 against the unmasked kernels), the first and
    the full head pass for every subset of {g_kl, g_scores, g_pooled}, and v = scores = NULL with g_pooled only."""
    li = LAYOUTS.index(layout)
    seed = 7 * D + 31 * li + KINDS.index(kind)
    pc = PairCase(layout, seed)
    P, R, N = pc.P, pc.R, pc.N
    x, hs32, gate, v, c, dist = _inputs(pc, dt, D)
    masked, sig = _masked(kind), kind.startswith("sig")
    p = DROP_P[li % 3] if masked else 0.0
    stream_id = 1 + li % 2
    M = drop_masks(pc, stream_id, p, D) if masked else None
    X32 = masked_rows(hs32, pc, M, dt)
    X = X32.astype(np.float64)
    h = wide_rows(x, dt)
    assert np.array_equal(h.float().cpu().numpy(), hs32)
    dist_d = i32(dist).long() if seed % 2 else i32(dist)       # both distance instantiations
    dist_d = dist_d if R else (torch.zeros(1, dtype=dist_d.dtype, device=DEV)[:0])
    c_null = li % 2 == 1
    gate_d, v_d, c_d = f32(gate), f32(v), (None if c_null else f32(c))
    E = ELEMS[dt]
    D_pad = -(-D // E) * E
    kw = dict(stream_id=stream_id, p=p)

    # ---- forward
    got = run_scores(kind, pc, h, gate_d, v_d, c_d, dist_d, **kw)
    want, bnd = pair_scores_ref(pc, X, gate.astype(np.float64), v.astype(np.float64),
                                np.zeros(P) if c_null else c.astype(np.float64), dist.astype(np.float64), D_pad,
                                sig=sig, dt=dt)
    for k, t in got.items():
        assert_within(host(t), want[k], bnd[k], f"scores pass: {k}")
    lean = run_scores(kind, pc, h, gate_d, v_d, c_d, dist_d, units=False, **kw)
    assert torch.equal(lean["scores"], got["scores"]) and torch.equal(lean["kl_b"], got["kl_b"])
    if masked and p == 0.0:                                   # the masked kernel at p = 0 is the unmasked one, bit for bit
        base = run_scores("plain" if kind == "drop" else "sig", pc, h, gate_d, v_d, c_d, dist_d)
        for k in base:
            assert torch.equal(base[k], got[k]), f"p = 0 vs unmasked: {k}"
    if P == 0:
        return _check_no_pairs(kind, pc, h, gate_d, v_d, dist_d, dt, D, kw)

    # ---- head backward, from the kernel's own scores and kl_b
    rng = pc.rng
    scores_d, klb_d = got["scores"], got["kl_b"]
    scores, klb = host(scores_d), host(klb_d)
    gs = rng.standard_normal(R).astype(np.float32)
    gp = rng.standard_normal((P, D)).astype(np.float32)
    arg_s = np.full((pc.S, D), -1, np.int64)                # the sentences' arg-max rows, -1 in some columns
    for s in range(pc.S):
        if pc.sp[s + 1] > pc.sp[s]:
            arg_s[s] = rng.integers(pc.sp[s], pc.sp[s + 1], D)
            arg_s[s, rng.random(D) < 0.2] = -1
    arg = arg_s
    if masked:                  # the final pool's per-pair arg-max rows: the sentence's at p = 0, each pair's own else
        arg = arg_s[pc.pair_sent]
        if p > 0:
            for q in range(P):
                s = pc.pair_sent[q]
                if pc.sp[s + 1] > pc.sp[s]:
                    arg[q] = rng.integers(pc.sp[s], pc.sp[s + 1], D)
    arg_x = pc.expanded_arg(arg, masked)
    mmax = np.where(arg_x >= 0, X32[np.maximum(arg_x, 0), np.arange(D)[None, :]] if R else 0, 0).astype(np.float32)
    gk = np.float32(0.7)
    dev_g = dict(g_kl=torch.tensor([float(gk)], dtype=torch.float32, device=DEV), g_scores=f32(gs), g_pooled=f32(gp),
                 arg=i32(arg), mmax=f32(mmax))
    dh_u = U_BF16 if dt == "bf16" else 0.0
    G, V64 = gate.astype(np.float64), v.astype(np.float64)
    # every subset of the gradient inputs, then v = scores = NULL with g_pooled only; the two layouts of more than
    # 10k pair rows run the empty and the full subset only, to keep the host references affordable
    subsets = GRAD_SUBSETS if R <= 10_000 else [(0, 0, 0), (1, 1, 1)]
    cases = [(a, b, q, False) for a, b, q in subsets] + [(0, 0, 1, True)]
    for kl_on, sc_on, p_on, no_v in cases:
        what = f"g_kl={kl_on} g_scores={sc_on} g_pooled={p_on}{' v=scores=NULL' if no_v else ''}"
        want, bnd = pair_head_ref(pc, X, M, G, np.zeros_like(V64) if no_v else V64, dist.astype(np.float64),
                                  scores, klb, float(gk) if kl_on else None, gs.astype(np.float64) if sc_on else None,
                                  gp.astype(np.float64) if p_on else None, arg_x if p_on else None, sig=sig, dt=dt)
        bnd["dh"] = bnd["dh"] + dh_u * (np.abs(want["dh"]) + bnd["dh"])      # the store rounds once to bf16
        for full_pass in (False, True):
            r = run_head(kind, pc, h, gate_d, None if no_v else v_d, dist_d, None if no_v else scores_d, klb_d,
                         dev_g["g_kl"] if kl_on else None, dev_g["g_scores"] if sc_on else None,
                         dev_g["g_pooled"] if p_on else None, dev_g["arg"] if p_on else None,
                         dev_g["mmax"] if p_on else None, full_pass, **kw)
            keys = ("dv", "dc") + (("dh", "dgate") if full_pass else ())
            for k in keys:
                assert_within(host(r[k]), want[k], bnd[k], f"{what} full_pass={full_pass}: {k}")
            if full_pass:
                pad = host(full(r["dh"])[:N, D:D_pad])             # the chain reads whole 16-byte chunks
                assert np.all(np.isfinite(pad)), f"{what}: dh padding"
            if masked and p == 0.0:
                base = run_head("plain" if kind == "drop" else "sig", pc, h, gate_d, None if no_v else v_d, dist_d,
                                None if no_v else scores_d, klb_d, dev_g["g_kl"] if kl_on else None,
                                dev_g["g_scores"] if sc_on else None, dev_g["g_pooled"] if p_on else None,
                                i32(arg_s) if p_on else None, None, full_pass)
                for k in keys:
                    assert_within(host(r[k]), host(base[k]), 2 * bnd[k], f"{what} p = 0 vs unmasked: {k}")


def _check_no_pairs(kind, pc, h, gate_d, v_d, dist_d, dt, D, kw):
    """P = 0 with rows present: the head backward writes d h = 0 (padding included) and nothing else."""
    for full_pass in (False, True):
        r = run_head(kind, pc, h, gate_d, v_d, dist_d, nan_f32(1)[:0], nan_f32(1)[:0], None, None, None, None, None,
                     full_pass, **kw)
        assert torch.isnan(r["ds_ws"]).all(), "ds_ws"
        for k in ("dv", "dc") + (("dgate",) if full_pass else ()):
            assert r[k].numel() == 0
        if full_pass:
            assert (full(r["dh"])[:pc.N] == 0).all(), "dh"


@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("dt", ["bf16", "f32"])
def test_scores_and_head_reject_past_128_chunks(kind, dt):
    """One 16-byte chunk past the limit (bf16 D = 1032, fp32 D = 1028): every scores and head-backward entry point
    raises and leaves its outputs at the sentinels."""
    L, _ = _L()
    D = PAST_LIMIT[dt]
    pc = PairCase("short", 5)
    x, hs32, gate, v, c, dist = _inputs(pc, dt, D)
    h = wide_rows(x, dt)
    kw = dict(stream_id=1, p=0.25)
    outs = {}
    with pytest.raises(L.EdgError, match="status"):
        run_scores(kind, pc, h, f32(gate), f32(v), f32(c), i32(dist), keep=outs, **kw)
    heads = {}
    arg = i32(np.repeat(pc.sp[pc.pair_sent if _masked(kind) else np.arange(pc.S)][:, None], D, 1))
    with pytest.raises(L.EdgError, match="status"):
        run_head(kind, pc, h, f32(gate), f32(v), i32(dist), nan_f32(pc.R), nan_f32(pc.P),
                 torch.ones(1, device=DEV), None, f32(np.ones((pc.P, D))), arg, nan_f32(pc.P, D), True, keep=heads, **kw)
    torch.cuda.synchronize()
    for k, t in list(outs.items()) + list(heads.items()):
        assert torch.isnan(t).all(), k


# ------------------------------------------------------------------------------------------------ the pool
POOL_VIEWS = (1, 2, 3, 4, 5)    # V = 5: a second launch, on streams stream0 + 4


def pool_reference(pc, hs32, gates, stream0, p, dt):
    """edg_pool_drop_pairs restated in fp32: view v reads its pair's rows under stream stream0 + v; the column maximum
    with its first row (strict >), pooled = the fp32 product m * g, arg = that row (the sentence's first row where
    g = 0), mmax = m; a pair of an empty sentence gives 0 / -1 / 0."""
    V, P, D = gates.shape
    pooled, mmax = np.zeros((V, P, D), np.float32), np.zeros((V, P, D), np.float32)
    arg = np.full((V, P, D), -1, np.int64)
    for v in range(V):
        Xv = masked_rows(hs32, pc, drop_masks(pc, stream0 + v, p, D), dt)
        for q in range(P):
            lo, hi = pc.prp[q], pc.prp[q + 1]
            if hi == lo:
                continue
            beg = pc.sp[pc.pair_sent[q]]
            m = Xv[lo:hi].max(0)
            g = gates[v, q]
            pooled[v, q], mmax[v, q] = m * g, m
            arg[v, q] = np.where(g != 0, beg + np.argmax(Xv[lo:hi] == m, axis=0), beg)
    return pooled, arg, mmax


@pytest.mark.gpu
@pytest.mark.parametrize("dt,D,layout", grid())
def test_pool_drop_pairs(dt, D, layout):
    """edg_pool_drop_pairs bit for bit against its rule on each pair's masked rows, V in 1 .. 5, stream0 in {0, 2} and
    p in {0, 0.25, 0.9} (at 0.9 whole columns drop: ties at 0 and arg-max rows that are dropped); at p = 0 it equals
    edg_pool_fwd on the expanded batch."""
    from test_gpu_i_staged_windows import run_pool as run_pool_sentences
    from ed_gated_gcn_b200 import ops
    li = LAYOUTS.index(layout)
    pc = PairCase(layout, 3 * D + li)
    rng, P = pc.rng, pc.P
    V, stream0 = POOL_VIEWS[(li + D) % 5], 2 * ((li + D // 4) % 2)
    x = rng.standard_normal((pc.N, D)).astype(np.float32)
    x[:, 5 % D] = -np.abs(x[:, 5 % D]) - 0.25                 # negative everywhere: a dropped 0 beats every kept row
    for s in range(0, pc.S, 2):                               # ties: a repeated row
        if pc.sp[s + 1] - pc.sp[s] > 1:
            x[pc.sp[s] + 1] = x[pc.sp[s]]
    hs32, h = to_T(x, dt), wide_rows(x, dt)
    gates = (rng.random((V, P, D)) + 0.05).astype(np.float32)
    gates[:, ::2, 3 % D] = 0.0
    gates_d = f32(gates)
    for p in DROP_P:
        pooled, arg, mmax = run_pool(pc, h, gates_d, stream0, p)
        want_p, want_a, want_m = pool_reference(pc, hs32, gates, stream0, p, dt)
        what = f"V={V} stream0={stream0} p={p}"
        assert np.array_equal(pooled.cpu().numpy().view(np.int32), want_p.view(np.int32)), f"{what}: pooled"
        assert np.array_equal(arg.cpu().numpy().astype(np.int64), want_a), f"{what}: arg"
        assert np.array_equal(mmax.cpu().numpy().view(np.int32), want_m.view(np.int32)), f"{what}: mmax"
        if p == 0.0 and P:
            g = types.SimpleNamespace(sent_ptr=i32(pc.prp), row_sent=None, n_rows=pc.R,
                                      max_len=int(np.diff(pc.prp).max()))
            hx = ops.as_rows(torch.from_numpy(hs32[pc.rows]).to(DEV), TORCH_DT[dt]) if pc.R else \
                ops.alloc_rows(0, D, TORCH_DT[dt], DEV, zero=True)
            sp_, sa, sh = run_pool_sentences(hx, g, gates_d.contiguous())
            assert torch.equal(sp_, pooled), "p = 0 vs edg_pool_fwd: pooled"
            assert all(torch.equal(sh, mmax[v]) for v in range(V)), "p = 0 vs edg_pool_fwd: mmax"
            sa = sa.cpu().numpy().astype(np.int64)
            back = np.where(sa >= 0, sa - pc.prp[:-1, None] + pc.sp[pc.pair_sent][:, None], -1)
            assert np.array_equal(back, want_a), "p = 0 vs edg_pool_fwd: arg"


# ------------------------------------------------------------------------------------------------ the views backward
def _call_views_hmax(pc, hmax, gates, g_xy, dgates, patch, acc_view):
    L, _ = _L()
    V, P, D = gates.shape
    L.call("edg_views_bwd_hmax_pairs", L.ptr(hmax), rows_ptr(gates), L.ptr(g_xy), V, pc.S, rows_ptr(pc.dev.pair_ptr), P,
           D, L.ptr(patch), patch.shape[1], rows_ptr(dgates), acc_view, L.stream())


@pytest.mark.gpu
@pytest.mark.parametrize("D,layout", [pytest.param(D, n, id=f"D{D}-{n}") for D in (20, 132, 300, 1024)
                                      for n in layouts_for(D)])
def test_views_bwd_hmax_pairs(D, layout):
    """edg_views_bwd_hmax_pairs against its fp32 formulas in fp64 with bounds of a few u, acc_view in {-1, 0, V - 1}
    onto d gates pre-filled with a known value, patch_val at a pitch wider than D (the columns past D untouched)."""
    li = LAYOUTS.index(layout)
    pc = PairCase(layout, 5 * D + li)
    rng, P, S = pc.rng, pc.P, pc.S
    V = (1, 2, 3)[li % 3]
    hmax = rng.standard_normal((S, D)).astype(np.float32)
    gates = rng.random((V, P, D)).astype(np.float32)
    gates[:, :, 3 % D] = 0.0
    gxy = np.float32(0.3)
    hm = hmax.astype(np.float64)[pc.pair_sent]                # [P,D]
    g = gates.astype(np.float64)
    gx = np.float64(gxy) / P if P else 0.0
    gsum, gabs = g.sum(0), np.abs(g).sum(0)
    dp = gx * (gsum[None] - g) * hm[None]
    edp = np.abs(gx * hm)[None] * (V + 1) * U * gabs[None] + 4 * U * np.abs(dp)
    dg = dp * hm[None]
    edg = edp * np.abs(hm)[None] + U * np.abs(dg)
    pv_terms = (dp * g).sum(0)
    want_pv = np.zeros((S, D))
    np.add.at(want_pv, pc.pair_sent, pv_terms)
    e_pv, mag = np.zeros((S, D)), np.zeros((S, D))
    np.add.at(e_pv, pc.pair_sent, (edp * np.abs(g) + U * np.abs(dp * g)).sum(0))
    np.add.at(mag, pc.pair_sent, np.abs(dp * g).sum(0))
    e_pv += (V * np.diff(pc.pp) + 1)[:, None] * U * mag
    gates_d = f32(gates)
    for acc_view in (-1, 0, V - 1):
        dgates = torch.full((V, max(P, 1), D), KEEP_PATTERN, dtype=torch.float32, device=DEV)
        patch = nan_f32(S, D + 4)
        _call_views_hmax(pc, f32(hmax), gates_d, torch.tensor([float(gxy)], device=DEV), dgates[:, :P], patch,
                         acc_view)
        acc = (np.arange(V) == acc_view)[:, None, None]
        want_dg = np.where(acc, KEEP_PATTERN + dg, dg)
        assert_within(host(dgates[:, :P]), want_dg, edg + acc * U * np.abs(want_dg), f"acc_view={acc_view}: dgates")
        assert_within(host(patch[:, :D]), want_pv, e_pv, f"acc_view={acc_view}: patch_val")
        assert torch.isnan(patch[:, D:]).all(), "patch_val past D"


def _call_views_drop(pc, pooled, mmax, arg, gates, g_xy, p, dh, dgates, acc_view):
    L, ops = _L()
    V, P, D = pooled.shape
    seed = torch.tensor([SEED], dtype=torch.int64, device=DEV)
    d = pc.dev
    L.call("edg_views_bwd_drop_pairs", rows_ptr(pooled), rows_ptr(mmax), rows_ptr(arg), rows_ptr(gates), L.ptr(g_xy), V,
           rows_ptr(d.sent_ptr), rows_ptr(d.row_sent) if pc.N else None, pc.N, rows_ptr(d.pair_ptr),
           rows_ptr(d.pair_row_ptr), P, D, L.ptr(seed), float(p), rows_ptr(dh), L.dt(dh), ops.ld(dh), rows_ptr(dgates),
           acc_view, L.stream())


@pytest.mark.gpu
@pytest.mark.parametrize("dt,D,layout", grid())
def test_views_bwd_drop_pairs(dt, D, layout):
    """edg_views_bwd_drop_pairs: d gates against the fp32 formula (fp64, bounds of a few u) with acc_view in
    {-1, 0, V - 1}; the views' share of d h_1 against the fp64 sum over the row's pairs and views of keep * scale *
    gate * dP (view v keyed on stream v at the pair's own row), added once into d h and rounded to T.  Every element
    no arg-max row reaches, padding columns included, comes back bit-unchanged."""
    from ed_gated_gcn_b200 import ops
    li = LAYOUTS.index(layout)
    pc = PairCase(layout, 11 * D + li)
    rng, P, N, R = pc.rng, pc.P, pc.N, pc.R
    V, p = (1, 2, 3, 4)[li % 4], DROP_P[(li + 1) % 3]
    pooled = rng.standard_normal((V, P, D)).astype(np.float32)
    mmax = rng.standard_normal((V, P, D)).astype(np.float32)
    gates = rng.random((V, P, D)).astype(np.float32)
    arg = np.full((V, P, D), -1, np.int64)
    for q in range(P):
        s = pc.pair_sent[q]
        if pc.sp[s + 1] > pc.sp[s]:
            arg[:, q] = rng.integers(pc.sp[s], pc.sp[s + 1], (V, D))
    gxy = np.float32(0.3)
    pooled_d, mmax_d, gates_d, arg_d = f32(pooled), f32(mmax), f32(gates), i32(arg)
    # fp64 references
    gx = np.float64(gxy) / P if P else 0.0
    pl, g = pooled.astype(np.float64), gates.astype(np.float64)
    tot, tabs = pl.sum(0), np.abs(pl).sum(0)
    dP = gx * (tot[None] - pl)
    edP = np.abs(gx) * (V + 1) * U * tabs[None] + 3 * U * np.abs(dP)
    dg = dP * mmax
    edg = edP * np.abs(mmax) + U * np.abs(dg)
    acc, eacc, mag = np.zeros((N, D)), np.zeros((N, D)), np.zeros((N, D))
    hits = np.zeros((N, D), np.int64)
    cols = np.broadcast_to(np.arange(D), (P, D))
    for v in range(V):
        M = drop_masks(pc, v, p, D)
        ok = arg[v] >= 0
        t = arg[v][ok]
        key = (pc.prp[:-1, None] + arg[v] - pc.sp[pc.pair_sent][:, None])[ok]
        term = M[key, cols[ok]] * g[v][ok] * dP[v][ok]
        np.add.at(acc, (t, cols[ok]), term)
        np.add.at(eacc, (t, cols[ok]), M[key, cols[ok]] * (g[v][ok] * edP[v][ok] + 3 * U * np.abs(term)))
        np.add.at(mag, (t, cols[ok]), np.abs(term))
        np.add.at(hits, (t, cols[ok]), 1)
    eacc += (hits + 1) * U * mag
    for acc_view in (-1, 0, V - 1):
        dh = ops.alloc_rows(N, D, TORCH_DT[dt], DEV)
        base = full(dh)
        base.copy_(torch.from_numpy(rng.standard_normal(tuple(base.shape)).astype(np.float32)).to(DEV))
        old = host(base)
        dgates = torch.full((V, max(P, 1), D), KEEP_PATTERN, dtype=torch.float32, device=DEV)
        _call_views_drop(pc, pooled_d, mmax_d, arg_d, gates_d, torch.tensor([float(gxy)], device=DEV), p, dh,
                         dgates[:, :P], acc_view)
        on = (np.arange(V) == acc_view)[:, None, None]
        want_dg = np.where(on, KEEP_PATTERN + dg, dg)
        what = f"V={V} p={p} acc_view={acc_view}"
        assert_within(host(dgates[:, :P]), want_dg, edg + on * U * np.abs(want_dg), f"{what}: dgates")
        got = host(base)
        want = old[:N, :D] + acc
        assert_within(got[:N, :D], want, eacc + U_T[dt] * np.abs(want) + U * np.abs(want), f"{what}: dh")
        same = np.ones_like(got, dtype=bool)
        same[:N, :D] = hits == 0
        assert np.array_equal(got[same], old[same]), f"{what}: rows no view reaches changed"


# ------------------------------------------------------------------------------------------------ d x at the triggers
@pytest.mark.gpu
@pytest.mark.parametrize("dt,D,layout", [a for a in grid() if a.values[2] not in ("empty_owner", "all_empty")])
def test_trigger_scatter_add_pairs(dt, D, layout):
    """edg_trigger_scatter_add_pairs bit for bit: dx[pair_start + anchor] += da + sum_k extra[k], the sum in fp32 in
    order and the add rounded to T once per pair, the pairs of a sentence in ascending order (repeated anchors see
    each other's roundings); da = NULL with extra, 0 / 1 / 2 extra terms; every other element unchanged."""
    L, ops = _L()
    li = LAYOUTS.index(layout)
    pc = PairCase(layout, 13 * D + li)
    rng, P, N = pc.rng, pc.P, pc.N
    n_extra = li % 3
    use_da = n_extra == 0 or li % 2 == 0
    da = rng.standard_normal((P, D)).astype(np.float32)
    extra = rng.standard_normal((n_extra, P, D)).astype(np.float32)
    dx = ops.alloc_rows(N, D, TORCH_DT[dt], DEV)
    base = full(dx)
    base.copy_(torch.from_numpy(rng.standard_normal(tuple(base.shape)).astype(np.float32) * 4).to(DEV))
    want = base.float().cpu().numpy()
    da_d, extra_d, d = (f32(da) if use_da else None), (f32(extra) if n_extra else None), pc.dev
    L.call("edg_trigger_scatter_add_pairs", rows_ptr(da_d), rows_ptr(extra_d), n_extra, pc.S, rows_ptr(d.pair_ptr), P,
           D, rows_ptr(d.pair_start), rows_ptr(d.anchor), L.ptr(dx), L.dt(dx), ops.ld(dx), L.stream())
    for q in range(P):                                        # pairs are grouped by sentence in ascending order
        val = da[q].copy() if use_da else np.zeros(D, np.float32)
        for k in range(n_extra):
            val = (val + extra[k, q]).astype(np.float32)
        r = pc.sp[pc.pair_sent[q]] + pc.anchor[q]
        want[r, :D] = to_T(want[r, :D] + val, dt)
    assert np.array_equal(base.float().cpu().numpy().view(np.int32), want.view(np.int32))
