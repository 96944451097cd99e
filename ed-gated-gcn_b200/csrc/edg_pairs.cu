// Every candidate trigger of a sentence from one pass of the GCN chain (include/edgcn.h, "Trigger pairs").
//
// The GCN chain h_1 .. h_L depends on the sentence and not on the trigger, so the rows of a sentence exist once, and
// only what depends on the trigger runs per (sentence, trigger) pair p: the scores / kl of bert_amir5.py:645-648 over
// the sentence's rows against that pair's g_p * v_p, and their backward.  The pairs of sentence s are the contiguous
// range pair_ptr[s] .. pair_ptr[s+1] - 1; per-pair row outputs (scores, dist, ...) live in the per-pair packed layout
// whose pair p starts at pair_row_ptr[p].  Every sum over the pairs of a sentence runs in ascending pair order inside
// one thread (no atomics), so the results do not depend on scheduling.
//
// Gate dropout (GatedGCNStack(pair_dropout=True)): pair p reads row t of its sentence under the mask the expanded batch
// applies to that row's copy, keep(seed, stream, pair_row_ptr[p] + t, column) -- every pair draws its own mask.  The
// masks are regenerated from the seed wherever they are needed; nothing is stored per (pair, row).
//
// Included after edg_block.cu (softmax_stats, dist_at, ScoresQ).

namespace edg {

// ---- row mask policies of the per-pair kernels --------------------------------------------------------------------
// NoMask: the rows as stored.  GateDrop: the gate-dropout mask of one stream; a kept element reads as
// T(h * scale) (the value edg_dropout_rows stores), a dropped one as 0.
struct NoMask {
  static constexpr bool kDrop = false;
  struct Key {};
  __device__ __forceinline__ Key key() const { return Key{}; }
  template <typename T, int E>
  __device__ __forceinline__ void apply(Key, float (&)[E], int, int) const {}
};
struct GateDrop {
  static constexpr bool kDrop = true;
  const int64_t* seed;       // device scalar
  uint32_t stream_id, thr;   // thr = dropout_threshold(p)
  float scale;               // 1 / (1 - p)
  const float* mmax;         // head backward: the pair's masked column maxima of h_L [P,D] (its pooled rows' values)
  using Key = DropKey;
  __device__ __forceinline__ Key key() const { return dropout_key(seed, stream_id); }
  __device__ __forceinline__ bool keep(Key k, int row, int col) const {
    return dropout_keep(k, (uint32_t)row, (uint32_t)col, thr);
  }
  template <typename T, int E>
  __device__ __forceinline__ void apply(Key k, float (&f)[E], int row, int c) const {
#pragma unroll
    for (int i = 0; i < E; ++i) f[i] = keep(k, row, c + i) ? to_f32(from_f32<T>(f[i] * scale)) : 0.f;
  }
};

// ---- scores, softmax product and d kl / d (v, c) units per pair -----------------------------------------
// One warp per pair (the per-pair twin of scores_kl_fwd_kernel): the sentence's rows are read through L1 / L2, where
// the consecutive pairs of a sentence -- consecutive warps of a block -- find them.
template <typename T, int I64, class Mask>
__global__ void __launch_bounds__(128)
scores_kl_pairs_kernel(const T* __restrict__ h, int64_t ldh, const int32_t* __restrict__ sent_ptr,
                       const int32_t* __restrict__ pair_sent, const int32_t* __restrict__ pair_row_ptr, int P, int D,
                       int chunks, const float* __restrict__ gate, const float* __restrict__ vvec,
                       const float* __restrict__ cvec, const void* __restrict__ dist, float* __restrict__ scores,
                       float* __restrict__ kl_b, float* __restrict__ dv_unit, float* __restrict__ dc_unit,
                       float* __restrict__ u_unit, float* __restrict__ sf_unit, Mask mask) {
  constexpr int E = Vec16<T>::kElems;
  constexpr int kMaxQ = ScoresQ<T>::value;
  const int p = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (p >= P) return;
  const int lane = threadIdx.x & 31;
  const int s = __ldg(pair_sent + p);
  const int beg = __ldg(sent_ptr + s), end = __ldg(sent_ptr + s + 1), n = end - beg;
  const int o0 = __ldg(pair_row_ptr + p);                 // this pair's rows in the per-pair layout
  const typename Mask::Key key = mask.key();
  float w[kMaxQ][E];
#pragma unroll
  for (int q = 0; q < kMaxQ; ++q) {
    const int c = (lane + 32 * q) * E;
#pragma unroll
    for (int k = 0; k < E; ++k)
      w[q][k] = (lane + 32 * q < chunks && c + k < D)
                    ? __ldg(gate + (int64_t)p * D + c + k) * __ldg(vvec + (int64_t)p * D + c + k) : 0.f;
  }
  const float cb = cvec ? __ldg(cvec + p) : 0.f;
  constexpr int U = 4;                        // rows in flight per warp
  for (int t = 0; t < n; t += U) {
    float sacc[U];
#pragma unroll
    for (int u = 0; u < U; ++u) sacc[u] = 0.f;
#pragma unroll
    for (int q = 0; q < kMaxQ; ++q) {
      if (lane + 32 * q < chunks) {
        float f[U][E];
#pragma unroll
        for (int u = 0; u < U; ++u)
          if (t + u < n) Vec16<T>::load(h + (int64_t)(beg + t + u) * ldh + (lane + 32 * q) * E, f[u]);
#pragma unroll
        for (int u = 0; u < U; ++u)
          if (t + u < n) {
            mask.template apply<T>(key, f[u], o0 + t + u, (lane + 32 * q) * E);
#pragma unroll
            for (int k = 0; k < E; ++k) sacc[u] = fmaf(f[u][k], w[q][k], sacc[u]);
          }
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) sacc[u] = warp_sum(sacc[u]);
    if (lane < U && t + lane < n) {
      float mine = sacc[0];
#pragma unroll
      for (int u = 1; u < U; ++u) mine = (lane == u) ? sacc[u] : mine;
      scores[o0 + t + lane] = mine + cb;
    }
  }
  __syncwarp();
  float ms, zs, mq, zq;
  softmax_stats<I64>(scores, dist, o0, o0 + n, lane, ms, zs, mq, zq);
  float acc = 0.f;
  for (int t = o0 + lane; t < o0 + n; t += 32)
    acc += (expf(scores[t] - ms) / zs) * (expf(dist_at<I64>(dist, t) - mq) / zq);
  acc = warp_sum(acc);
  if (lane == 0) kl_b[p] = acc;
  if (dv_unit == nullptr) return;
  // u_t = P_t (Q_t - kl_b) / P,  dv_unit = g * sum_t u_t h_t,  dc_unit = sum_t u_t  (kl is the mean over the P pairs)
  const float klb = acc, invP = 1.0f / (float)P;
  float dvu[kMaxQ][E];
#pragma unroll
  for (int q = 0; q < kMaxQ; ++q)
#pragma unroll
    for (int k = 0; k < E; ++k) dvu[q][k] = 0.f;
  float dcu = 0.f;
  for (int t = 0; t < n; ++t) {
    const float u = (expf(scores[o0 + t] - ms) / zs) * ((expf(dist_at<I64>(dist, o0 + t) - mq) / zq) - klb) * invP;
    dcu += u;
    if (lane == 0 && u_unit) u_unit[o0 + t] = u;
#pragma unroll
    for (int q = 0; q < kMaxQ; ++q) {
      if (lane + 32 * q < chunks) {
        float f[E];
        Vec16<T>::load(h + (int64_t)(beg + t) * ldh + (lane + 32 * q) * E, f);
        mask.template apply<T>(key, f, o0 + t, (lane + 32 * q) * E);
#pragma unroll
        for (int k = 0; k < E; ++k) dvu[q][k] = fmaf(u, f[k], dvu[q][k]);
      }
    }
  }
#pragma unroll
  for (int q = 0; q < kMaxQ; ++q) {
    const int c = (lane + 32 * q) * E;
#pragma unroll
    for (int k = 0; k < E; ++k)
      if (lane + 32 * q < chunks && c + k < D) {
        dv_unit[(int64_t)p * D + c + k] = dvu[q][k] * __ldg(gate + (int64_t)p * D + c + k);
        if (sf_unit) sf_unit[(int64_t)p * D + c + k] = dvu[q][k];
      }
  }
  if (lane == 0 && dc_unit) dc_unit[p] = dcu;
}

// ---- head backward, per-pair part: ds, dc, dv, dgate ----------------------------------------------------
// One warp per pair.  ds_t = g_kl / P * P_t (Q_t - kl_b) + g_scores_t goes to the workspace (the row pass below reads
// it); with sf = sum_t ds_t h_t:  dv = g * sf,  dc = sum_t ds_t,  dgate = v * sf + g_pooled * h[arg].
// Under GateDrop h_t is the pair's masked row and h[arg] its masked column maximum (mask.mmax).
template <typename T, int I64, class Mask>
__global__ void __launch_bounds__(128)
head_pairs_kernel(const T* __restrict__ h, int64_t ldh, const int32_t* __restrict__ sent_ptr,
                  const int32_t* __restrict__ pair_sent, const int32_t* __restrict__ pair_row_ptr, int P, int D, int chunks,
                  const float* __restrict__ gate, const float* __restrict__ vvec, const void* __restrict__ dist,
                  const float* __restrict__ scores, const float* __restrict__ kl_b, const float* __restrict__ g_kl,
                  const float* __restrict__ g_scores, const float* __restrict__ g_pooled, const int32_t* __restrict__ arg,
                  float* __restrict__ ds_ws, float* __restrict__ dgate, float* __restrict__ dv, float* __restrict__ dc,
                  Mask mask) {
  constexpr int E = Vec16<T>::kElems;
  constexpr int kMaxQ = ScoresQ<T>::value;
  const int p = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (p >= P) return;
  const int lane = threadIdx.x & 31;
  const int s = __ldg(pair_sent + p);
  const int beg = __ldg(sent_ptr + s), end = __ldg(sent_ptr + s + 1), n = end - beg;
  const int o0 = __ldg(pair_row_ptr + p);
  const typename Mask::Key key = mask.key();
  const bool have_s = (scores != nullptr) && (g_kl != nullptr || g_scores != nullptr);
  float tot = 0.f;
  if (have_s) {
    float ms = 0.f, zs = 1.f, mq = 0.f, zq = 1.f;
    const float gk = g_kl ? (__ldg(g_kl) / (float)P) : 0.f;
    if (g_kl) softmax_stats<I64>(scores, dist, o0, o0 + n, lane, ms, zs, mq, zq);
    const float klb = g_kl ? kl_b[p] : 0.f;
    for (int t = o0 + lane; t < o0 + n; t += 32) {
      float v = 0.f;
      if (g_kl) {
        const float Pt = expf(scores[t] - ms) / zs, Qt = expf(dist_at<I64>(dist, t) - mq) / zq;
        v = gk * Pt * (Qt - klb);
      }
      if (g_scores) v += g_scores[t];
      ds_ws[t] = v;
      tot += v;
    }
    tot = warp_sum(tot);
  } else {
    for (int t = o0 + lane; t < o0 + n; t += 32) ds_ws[t] = 0.f;
  }
  if (lane == 0 && dc) dc[p] = tot;
  if (!dv && !dgate) return;
  __syncwarp();                               // ds_ws of every lane is visible to the whole warp
  float sf[kMaxQ][E];
#pragma unroll
  for (int q = 0; q < kMaxQ; ++q)
#pragma unroll
    for (int k = 0; k < E; ++k) sf[q][k] = 0.f;
  if (have_s) {
    for (int t = 0; t < n; ++t) {
      const float dst = ds_ws[o0 + t];
#pragma unroll
      for (int q = 0; q < kMaxQ; ++q) {
        if (lane + 32 * q < chunks) {
          float f[E];
          Vec16<T>::load(h + (int64_t)(beg + t) * ldh + (lane + 32 * q) * E, f);
          mask.template apply<T>(key, f, o0 + t, (lane + 32 * q) * E);
#pragma unroll
          for (int k = 0; k < E; ++k) sf[q][k] = fmaf(dst, f[k], sf[q][k]);
        }
      }
    }
  }
#pragma unroll
  for (int q = 0; q < kMaxQ; ++q) {
    const int c = (lane + 32 * q) * E;
#pragma unroll
    for (int k = 0; k < E; ++k)
      if (lane + 32 * q < chunks && c + k < D) {
        const int64_t o = (int64_t)p * D + c + k;
        if (dv) dv[o] = __ldg(gate + o) * sf[q][k];
        if (dgate) {
          float dg = vvec ? __ldg(vvec + o) * sf[q][k] : 0.f;
          if (g_pooled) {
            if constexpr (Mask::kDrop) {
              dg = fmaf(__ldg(g_pooled + o), __ldg(mask.mmax + o), dg);
            } else {
              const int r = __ldg(arg + (int64_t)s * D + c + k);
              if (r >= beg && r < end) dg = fmaf(__ldg(g_pooled + o), to_f32(h[(int64_t)r * ldh + c + k]), dg);
            }
          }
          dgate[o] = dg;
        }
      }
  }
}

// ---- head backward, row part: d h_L over the sentence rows ----------------------------------------------------
// thread = (row, 16-byte column chunk):  dh_t = sum_p ds_{p,t} (g_p v_p)  +  [t = arg_s] sum_p g_p g_pooled_p,
// the pairs of the row's sentence in ascending order.  Every row is written (0 where the sentence has no pairs).
// Under GateDrop each pair's term is multiplied by its mask (keep / (1 - p), regenerated per element) and the arg-max
// rows are the pair's own ([P,D]):  dh_t = sum_p keep_{p,t} s (ds_{p,t} g_p v_p + [t = arg_p] g_p g_pooled_p).
template <typename T, class Mask>
__global__ void __launch_bounds__(128)
dh_pairs_kernel(const int32_t* __restrict__ sent_ptr, const int32_t* __restrict__ row_sent,
                const int32_t* __restrict__ pair_ptr, const int32_t* __restrict__ pair_row_ptr, int N, int D, int chunks,
                const float* __restrict__ gate, const float* __restrict__ vvec, const float* __restrict__ g_pooled,
                const int32_t* __restrict__ arg, const float* __restrict__ ds_ws, int have_s, T* __restrict__ dh,
                int64_t lddh, Mask mask) {
  constexpr int E = Vec16<T>::kElems;
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int t = (int)(idx / chunks);
  if (t >= N) return;
  const int c = (int)(idx - (int64_t)t * chunks) * E;
  const int s = __ldg(row_sent + t);
  const int loc = t - __ldg(sent_ptr + s);
  const int p0 = __ldg(pair_ptr + s), p1 = __ldg(pair_ptr + s + 1);
  if constexpr (Mask::kDrop) {
    const typename Mask::Key key = mask.key();
    float o[E];
#pragma unroll
    for (int k = 0; k < E; ++k) o[k] = 0.f;
    for (int p = p0; p < p1; ++p) {
      const int64_t po = (int64_t)p * D + c;
      const int rk = __ldg(pair_row_ptr + p) + loc;             // this row's key in pair p's copy of the sentence
      const float dst = have_s ? __ldg(ds_ws + rk) : 0.f;
#pragma unroll
      for (int k = 0; k < E; ++k)
        if (c + k < D) {
          const float g = __ldg(gate + po + k);
          float term = have_s ? dst * (g * __ldg(vvec + po + k)) : 0.f;
          if (g_pooled && __ldg(arg + po + k) == t) term = fmaf(g, __ldg(g_pooled + po + k), term);
          if (mask.keep(key, rk, c + k)) o[k] = fmaf(mask.scale, term, o[k]);
        }
    }
    Vec16<T>::store(dh + (int64_t)t * lddh + c, o);
    return;
  }
  bool hit = false;                                   // this row is the arg-max row of one of the chunk's columns
  int32_t where[E];
#pragma unroll
  for (int k = 0; k < E; ++k) {
    where[k] = (g_pooled && c + k < D) ? __ldg(arg + (int64_t)s * D + c + k) : -1;
    hit |= where[k] == t;
  }
  float o[E], argsum[E];
#pragma unroll
  for (int k = 0; k < E; ++k) { o[k] = 0.f; argsum[k] = 0.f; }
  for (int p = p0; p < p1; ++p) {
    const int64_t po = (int64_t)p * D + c;
    if (have_s) {
      const float dst = __ldg(ds_ws + __ldg(pair_row_ptr + p) + loc);
#pragma unroll
      for (int k = 0; k < E; ++k)
        if (c + k < D) o[k] = fmaf(dst, __ldg(gate + po + k) * __ldg(vvec + po + k), o[k]);
    }
    if (hit) {
#pragma unroll
      for (int k = 0; k < E; ++k)
        if (c + k < D) argsum[k] = fmaf(__ldg(gate + po + k), __ldg(g_pooled + po + k), argsum[k]);
    }
  }
#pragma unroll
  for (int k = 0; k < E; ++k)
    if (where[k] == t) o[k] += argsum[k];
  Vec16<T>::store(dh + (int64_t)t * lddh + c, o);
}

// ---- backward of the pooled views + diversity term, per pair, from the sentence's column maxima ----------------
// thread = (sentence, column).  Pair p's views are g_{v,p} * hmax_s (positive gates share the arg-max row), so
//   d pooled_{v,p} = g_xy / P * (sum_{v'} g_{v',p} - g_{v,p}) * hmax_s,   d g_{v,p} = d pooled_{v,p} * hmax_s,
//   patch_val[s] = sum_p sum_v g_{v,p} d pooled_{v,p}   (what the arg-max row of d h_1 receives)
__global__ void __launch_bounds__(256)
views_bwd_hmax_pairs_kernel(const float* __restrict__ hmax, const float* __restrict__ gates, const float* __restrict__ g_xy,
                            int V, int S, const int32_t* __restrict__ pair_ptr, int P, int D, float* __restrict__ patch_val,
                            int64_t ldp, float* __restrict__ dgates, int acc_view) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (int64_t)S * D) return;
  const int s = (int)(i / D), d = (int)(i - (int64_t)s * D);
  const int64_t PD = (int64_t)P * D;
  const float gxy = g_xy ? (__ldg(g_xy) / (float)P) : 0.f;
  const float hm = hmax[i];
  float pval = 0.f;
  for (int p = __ldg(pair_ptr + s); p < __ldg(pair_ptr + s + 1); ++p) {
    const int64_t o = (int64_t)p * D + d;
    float gsum = 0.f;
    for (int v = 0; v < V; ++v) gsum += gates[v * PD + o];
    for (int v = 0; v < V; ++v) {
      const float g = gates[v * PD + o];
      const float dp = gxy * (gsum - g) * hm;
      pval = fmaf(dp, g, pval);
      const float dg = dp * hm;
      dgates[v * PD + o] = (v == acc_view) ? dgates[v * PD + o] + dg : dg;
    }
  }
  patch_val[(int64_t)s * ldp + d] = pval;
}

// ---- gated max-pool per pair under gate dropout ----------------------------------------------------------------
// thread = (pair, 16-byte column chunk), pool_fwd_kernel's rule on the pair's masked rows: view v reads its sentence's
// rows under the mask of stream drop.stream_id + v, all V views from one read of each row.  Column maximum m with its
// first row (strict >), pooled = m * g, arg = the row (beg where g == 0), mmax = m; an empty sentence gives 0 / -1 / 0.
template <typename T, int V>
__global__ void __launch_bounds__(128)
pool_drop_pairs_kernel(const T* __restrict__ h, int64_t ldh, const int32_t* __restrict__ sent_ptr,
                       const int32_t* __restrict__ pair_sent, const int32_t* __restrict__ pair_row_ptr, int P, int D,
                       int chunks, const float* __restrict__ gates, GateDrop drop, float* __restrict__ pooled,
                       int32_t* __restrict__ arg, float* __restrict__ mmax) {
  constexpr int E = Vec16<T>::kElems;
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int p = (int)(idx / chunks);
  if (p >= P) return;
  const int c = (int)(idx - (int64_t)p * chunks) * E;
  const int s = __ldg(pair_sent + p);
  const int beg = __ldg(sent_ptr + s), end = __ldg(sent_ptr + s + 1);
  const int rk0 = __ldg(pair_row_ptr + p) - beg;           // key of sentence row t in pair p's copy: rk0 + t
  DropKey key[V];
#pragma unroll
  for (int v = 0; v < V; ++v) key[v] = dropout_key(drop.seed, drop.stream_id + v);
  float m[V][E];
  int32_t where[V][E];
#pragma unroll
  for (int v = 0; v < V; ++v)
#pragma unroll
    for (int k = 0; k < E; ++k) { m[v][k] = -INFINITY; where[v][k] = beg; }
  constexpr int U = 2;                        // rows in flight per thread
  for (int t = beg; t < end; t += U) {
    float f[U][E];
#pragma unroll
    for (int u = 0; u < U; ++u)
      if (t + u < end) Vec16<T>::load(h + (int64_t)(t + u) * ldh + c, f[u]);
#pragma unroll
    for (int u = 0; u < U; ++u) {
      if (t + u >= end) break;
#pragma unroll
      for (int v = 0; v < V; ++v)
#pragma unroll
        for (int k = 0; k < E; ++k) {
          const float x = dropout_keep(key[v], (uint32_t)(rk0 + t + u), (uint32_t)(c + k), drop.thr)
                              ? to_f32(from_f32<T>(f[u][k] * drop.scale)) : 0.f;
          if (x > m[v][k]) { m[v][k] = x; where[v][k] = t + u; }      // strict: first row wins ties
        }
    }
  }
  const int64_t PD = (int64_t)P * D;
#pragma unroll
  for (int v = 0; v < V; ++v)
#pragma unroll
    for (int k = 0; k < E; ++k)
      if (c + k < D) {
        const int64_t o = v * PD + (int64_t)p * D + c + k;
        const float g = __ldg(gates + o);
        pooled[o] = (beg < end) ? m[v][k] * g : 0.f;
        arg[o] = (beg < end) ? (g != 0.f ? where[v][k] : beg) : -1;
        mmax[o] = (beg < end) ? m[v][k] : 0.f;
      }
}

// ---- backward of the pooled views + diversity term under gate dropout ---------------------------------------------
// dP_{v,p} = g_xy / P * (sum_{v'} pooled_{v',p} - pooled_{v,p}).  d gates, thread = (pair, column):
//   dgates[v,p] (+)= dP_{v,p} * mmax_{v,p}      (acc_view already holds d gate_L)
__global__ void __launch_bounds__(256)
views_dgates_drop_pairs_kernel(const float* __restrict__ pooled, const float* __restrict__ mmax,
                               const float* __restrict__ g_xy, int V, int P, int D, float* __restrict__ dgates,
                               int acc_view) {
  const int64_t PD = (int64_t)P * D;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= PD) return;
  const float gxy = g_xy ? (__ldg(g_xy) / (float)P) : 0.f;
  float tot = 0.f;
  for (int v = 0; v < V; ++v) tot += pooled[v * PD + i];
  for (int v = 0; v < V; ++v) {
    const float dg = gxy * (tot - pooled[v * PD + i]) * mmax[v * PD + i];
    dgates[v * PD + i] = (v == acc_view) ? dgates[v * PD + i] + dg : dg;
  }
}

// the views' share of d h_1, thread = (row, 16-byte column chunk), the row's pairs and then the views in ascending
// order, summed in fp32 and added to dh once:  dh_t += sum_p sum_v [t = arg_{v,p}] keep_{v,p,t} s gates_{v,p} dP_{v,p}
template <typename T>
__global__ void __launch_bounds__(128)
views_dh_drop_pairs_kernel(const float* __restrict__ pooled, const int32_t* __restrict__ arg,
                           const float* __restrict__ gates, const float* __restrict__ g_xy, int V,
                           const int32_t* __restrict__ sent_ptr, const int32_t* __restrict__ row_sent,
                           const int32_t* __restrict__ pair_ptr, const int32_t* __restrict__ pair_row_ptr, int N, int P,
                           int D, int chunks, GateDrop drop, T* __restrict__ dh, int64_t lddh) {
  constexpr int E = Vec16<T>::kElems;
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int t = (int)(idx / chunks);
  if (t >= N) return;
  const int c = (int)(idx - (int64_t)t * chunks) * E;
  const int s = __ldg(row_sent + t);
  const int loc = t - __ldg(sent_ptr + s);
  const int p0 = __ldg(pair_ptr + s), p1 = __ldg(pair_ptr + s + 1);
  const int64_t PD = (int64_t)P * D;
  const float gxy = g_xy ? (__ldg(g_xy) / (float)P) : 0.f;
  const DropKey key0 = dropout_key(drop.seed, 0);          // view v's key: lo ^ v * 0xC2B2AE3D (dropout_key)
  float acc[E];
  bool hit = false;
#pragma unroll
  for (int k = 0; k < E; ++k) {                            // one column at a time: little live state
    acc[k] = 0.f;
    if (c + k >= D) continue;
    for (int p = p0; p < p1; ++p) {
      const int64_t pk = (int64_t)p * D + c + k;
      for (int v = 0; v < V; ++v) {
        if (__ldg(arg + v * PD + pk) != t) continue;
        hit = true;
        float tot = 0.f;
        for (int w = 0; w < V; ++w) tot += __ldg(pooled + w * PD + pk);
        const float dp = gxy * (tot - __ldg(pooled + v * PD + pk));
        const DropKey kv{key0.lo ^ ((uint32_t)v * 0xC2B2AE3DU), key0.hi};
        if (dropout_keep(kv, (uint32_t)(__ldg(pair_row_ptr + p) + loc), (uint32_t)(c + k), drop.thr))
          acc[k] = fmaf(drop.scale, __ldg(gates + v * PD + pk) * dp, acc[k]);
      }
    }
  }
  if (!hit) return;
  T* q = dh + (int64_t)t * lddh + c;
  float o[E];
  Vec16<T>::load(q, o);
#pragma unroll
  for (int k = 0; k < E; ++k) o[k] += acc[k];
  Vec16<T>::store(q, o);
}

// ---- d x at the trigger rows, per pair ----------------------------------------------------------------------
// thread = (sentence, column): dx[pair_start[p] + anchor[p]] += da[p] + sum_k extra[k, p] for the sentence's pairs in
// ascending order.  Pairs may share an anchor row; one thread owns all of them.
template <typename T>
__global__ void trigger_scatter_add_pairs_kernel(const float* __restrict__ da, const float* __restrict__ extra, int n_extra,
                                                 int S, const int32_t* __restrict__ pair_ptr, int P, int D,
                                                 const int32_t* __restrict__ pair_start, const int32_t* __restrict__ anchor,
                                                 T* __restrict__ dx, int64_t lddx) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (int64_t)S * D) return;
  const int s = (int)(i / D), d = (int)(i - (int64_t)s * D);
  const int64_t PD = (int64_t)P * D;
  for (int p = __ldg(pair_ptr + s); p < __ldg(pair_ptr + s + 1); ++p) {
    const int64_t e = (int64_t)p * D + d;
    float v = da ? da[e] : 0.f;
    for (int k = 0; k < n_extra; ++k) v += extra[k * PD + e];
    T* q = dx + ((int64_t)__ldg(pair_start + p) + __ldg(anchor + p)) * lddx + d;
    *q = from_f32<T>(to_f32(*q) + v);
  }
}

}  // namespace edg

using namespace edg;

namespace edg {

template <class Mask>
static int scores_kl_pairs_launch(const void* h, int dtype, int64_t ldh, const int32_t* sent_ptr, const int32_t* pair_sent,
                                  const int32_t* pair_row_ptr, int32_t P, int32_t D, const float* gate, const float* v,
                                  const float* c, const void* dist, int dist_i64, float* scores, float* kl_b,
                                  float* dv_unit, float* dc_unit, float* u_unit, float* sf_unit, Mask mask,
                                  edg_stream stream) {
  if (P < 0 || D <= 0) return EDG_ERR_ARG;
  if (P == 0) return EDG_OK;
  if (!h || !sent_ptr || !pair_sent || !pair_row_ptr || !gate || !v || !dist || !scores || !kl_b) return EDG_ERR_ARG;
  if ((u_unit || sf_unit) && !dv_unit) return EDG_ERR_ARG;
  if (!aligned16(h) || !row_pitch_ok(dtype, ldh)) return EDG_ERR_ALIGN;
  cudaStream_t s = (cudaStream_t)stream;
  const unsigned blocks = (unsigned)((P + 3) / 4);
  EDG_DISPATCH_T(dtype, {
    constexpr int E = Vec16<T>::kElems;
    const int chunks = (D + E - 1) / E;
    if (chunks > 32 * ScoresQ<T>::value) return EDG_ERR_UNSUPPORTED;
    if (dist_i64)
      scores_kl_pairs_kernel<T, 1><<<blocks, 128, 0, s>>>((const T*)h, ldh, sent_ptr, pair_sent, pair_row_ptr, P, D, chunks,
                                                          gate, v, c, dist, scores, kl_b, dv_unit, dc_unit, u_unit, sf_unit,
                                                          mask);
    else
      scores_kl_pairs_kernel<T, 0><<<blocks, 128, 0, s>>>((const T*)h, ldh, sent_ptr, pair_sent, pair_row_ptr, P, D, chunks,
                                                          gate, v, c, dist, scores, kl_b, dv_unit, dc_unit, u_unit, sf_unit,
                                                          mask);
  })
  return check_launch();
}

template <class Mask>
static int head_bwd_pairs_launch(const void* h, int dtype, int64_t ldh, const int32_t* sent_ptr, int32_t S,
                                 const int32_t* row_sent, int32_t N, const int32_t* pair_ptr, const int32_t* pair_sent,
                                 const int32_t* pair_row_ptr, int32_t P, int32_t D, const float* gate, const float* v,
                                 const void* dist, int dist_i64, const float* scores, const float* kl_b, const float* g_kl,
                                 const float* g_scores, const float* g_pooled, const int32_t* arg, void* dh, int64_t lddh,
                                 float* dgate, float* dv, float* dc, float* ds_ws, Mask mask, edg_stream stream) {
  if (S < 0 || P < 0 || D <= 0) return EDG_ERR_ARG;
  if (!sent_ptr || !pair_ptr || !pair_row_ptr || !h || !ds_ws) return EDG_ERR_ARG;
  if (!dh && !dv && !dc) return P == 0 ? EDG_OK : EDG_ERR_ARG;
  if (dh && (N < 0 || (N > 0 && !row_sent))) return EDG_ERR_ARG;
  if (P > 0) {            // the per-pair arrays; with no pairs they are empty (may be NULL) and only dh = 0 is written
    if (!pair_sent || !gate || (dh && !dgate)) return EDG_ERR_ARG;
    if (g_pooled && !arg) return EDG_ERR_ARG;
    if ((g_kl || g_scores) && (!scores || !v)) return EDG_ERR_ARG;
    if (g_kl && (!dist || !kl_b)) return EDG_ERR_ARG;
  }
  if (!aligned16(h) || !row_pitch_ok(dtype, ldh)) return EDG_ERR_ALIGN;
  if (dh && (!aligned16(dh) || !row_pitch_ok(dtype, lddh))) return EDG_ERR_ALIGN;
  cudaStream_t s = (cudaStream_t)stream;
  const int have_s = (scores != nullptr) && (g_kl != nullptr || g_scores != nullptr);
  EDG_DISPATCH_T(dtype, {
    constexpr int E = Vec16<T>::kElems;
    const int chunks = (D + E - 1) / E;
    if (chunks > 32 * ScoresQ<T>::value) return EDG_ERR_UNSUPPORTED;
    if (P > 0) {
      const unsigned blocks = (unsigned)((P + 3) / 4);
      if (dist_i64)
        head_pairs_kernel<T, 1><<<blocks, 128, 0, s>>>((const T*)h, ldh, sent_ptr, pair_sent, pair_row_ptr, P, D, chunks, gate,
                                                       v, dist, scores, kl_b, g_kl, g_scores, g_pooled, arg, ds_ws, dgate, dv, dc,
                                                       mask);
      else
        head_pairs_kernel<T, 0><<<blocks, 128, 0, s>>>((const T*)h, ldh, sent_ptr, pair_sent, pair_row_ptr, P, D, chunks, gate,
                                                       v, dist, scores, kl_b, g_kl, g_scores, g_pooled, arg, ds_ws, dgate, dv, dc,
                                                       mask);
    }
    if (dh && N > 0) {
      const unsigned blocks = (unsigned)(((int64_t)N * chunks + 127) / 128);
      dh_pairs_kernel<T><<<blocks, 128, 0, s>>>(sent_ptr, row_sent, pair_ptr, pair_row_ptr, N, D, chunks, gate, v, g_pooled,
                                                arg, ds_ws, have_s, (T*)dh, lddh, mask);
    }
  })
  return check_launch();
}

// the pairs' dropout entry points: p in [0, 1), seed a device int64 scalar
static int gate_drop(const int64_t* seed, int32_t stream_id, float p, const float* mmax, GateDrop& m) {
  if (!seed || stream_id < 0 || !dropout_p_ok(p)) return EDG_ERR_ARG;
  m = GateDrop{seed, (uint32_t)stream_id, dropout_threshold(p), 1.0f / (1.0f - p), mmax};
  return EDG_OK;
}

}  // namespace edg

extern "C" int edg_scores_kl_pairs_fwd(const void* h, int dtype, int64_t ldh, const int32_t* sent_ptr,
                                       const int32_t* pair_sent, const int32_t* pair_row_ptr, int32_t P, int32_t D,
                                       const float* gate, const float* v, const float* c, const void* dist, int dist_i64,
                                       float* scores, float* kl_b, float* dv_unit, float* dc_unit, float* u_unit,
                                       float* sf_unit, edg_stream stream) {
  return scores_kl_pairs_launch(h, dtype, ldh, sent_ptr, pair_sent, pair_row_ptr, P, D, gate, v, c, dist, dist_i64, scores,
                                kl_b, dv_unit, dc_unit, u_unit, sf_unit, NoMask{}, stream);
}

extern "C" int edg_scores_kl_drop_pairs_fwd(const void* h, int dtype, int64_t ldh, const int32_t* sent_ptr,
                                            const int32_t* pair_sent, const int32_t* pair_row_ptr, int32_t P, int32_t D,
                                            const float* gate, const float* v, const float* c, const void* dist,
                                            int dist_i64, float* scores, float* kl_b, float* dv_unit, float* dc_unit,
                                            float* u_unit, float* sf_unit, const int64_t* seed, int32_t stream_id, float p,
                                            edg_stream stream) {
  GateDrop m;
  if (P < 0 || D <= 0) return EDG_ERR_ARG;
  if (P == 0) return EDG_OK;
  if (const int rc = gate_drop(seed, stream_id, p, nullptr, m)) return rc;
  return scores_kl_pairs_launch(h, dtype, ldh, sent_ptr, pair_sent, pair_row_ptr, P, D, gate, v, c, dist, dist_i64, scores,
                                kl_b, dv_unit, dc_unit, u_unit, sf_unit, m, stream);
}

extern "C" int edg_head_bwd_pairs(const void* h, int dtype, int64_t ldh, const int32_t* sent_ptr, int32_t S,
                                  const int32_t* row_sent, int32_t N, const int32_t* pair_ptr, const int32_t* pair_sent, const int32_t* pair_row_ptr, int32_t P,
                                  int32_t D, const float* gate, const float* v, const void* dist, int dist_i64,
                                  const float* scores, const float* kl_b, const float* g_kl, const float* g_scores,
                                  const float* g_pooled, const int32_t* arg, void* dh, int64_t lddh, float* dgate,
                                  float* dv, float* dc, float* ds_ws, edg_stream stream) {
  return head_bwd_pairs_launch(h, dtype, ldh, sent_ptr, S, row_sent, N, pair_ptr, pair_sent, pair_row_ptr, P, D, gate, v,
                               dist, dist_i64, scores, kl_b, g_kl, g_scores, g_pooled, arg, dh, lddh, dgate, dv, dc, ds_ws,
                               NoMask{}, stream);
}

extern "C" int edg_head_bwd_drop_pairs(const void* h, int dtype, int64_t ldh, const int32_t* sent_ptr, int32_t S,
                                       const int32_t* row_sent, int32_t N, const int32_t* pair_ptr,
                                       const int32_t* pair_sent, const int32_t* pair_row_ptr, int32_t P, int32_t D,
                                       const float* gate, const float* v, const void* dist, int dist_i64,
                                       const float* scores, const float* kl_b, const float* g_kl, const float* g_scores,
                                       const float* g_pooled, const int32_t* arg, const float* mmax, void* dh,
                                       int64_t lddh, float* dgate, float* dv, float* dc, float* ds_ws,
                                       const int64_t* seed, int32_t stream_id, float p, edg_stream stream) {
  GateDrop m;
  if (P > 0 && g_pooled && !mmax) return EDG_ERR_ARG;
  if (const int rc = gate_drop(seed, stream_id, p, mmax, m)) return rc;
  return head_bwd_pairs_launch(h, dtype, ldh, sent_ptr, S, row_sent, N, pair_ptr, pair_sent, pair_row_ptr, P, D, gate, v,
                               dist, dist_i64, scores, kl_b, g_kl, g_scores, g_pooled, arg, dh, lddh, dgate, dv, dc, ds_ws,
                               m, stream);
}

extern "C" int edg_pool_drop_pairs(const void* h, int dtype, int64_t ldh, const int32_t* sent_ptr, const int32_t* pair_sent,
                                   const int32_t* pair_row_ptr, int32_t P, int32_t D, const float* gates, int32_t V,
                                   const int64_t* seed, int32_t stream0, float p, float* pooled, int32_t* arg,
                                   float* mmax, edg_stream stream) {
  if (P < 0 || D <= 0 || V <= 0) return EDG_ERR_ARG;
  if (P == 0) return EDG_OK;
  if (!h || !sent_ptr || !pair_sent || !pair_row_ptr || !gates || !pooled || !arg || !mmax) return EDG_ERR_ARG;
  if (!aligned16(h) || !row_pitch_ok(dtype, ldh)) return EDG_ERR_ALIGN;
  GateDrop m;
  if (const int rc = gate_drop(seed, stream0, p, nullptr, m)) return rc;
  cudaStream_t s = (cudaStream_t)stream;
  const int64_t PD = (int64_t)P * D;
  EDG_DISPATCH_T(dtype, {
    constexpr int E = Vec16<T>::kElems;
    const int chunks = (D + E - 1) / E;
    const unsigned blocks = (unsigned)(((int64_t)P * chunks + 127) / 128);
    for (int v0 = 0; v0 < V; v0 += 4) {             // up to four views per read of the rows
      GateDrop mv = m;
      mv.stream_id = m.stream_id + (uint32_t)v0;
      const float* g = gates + v0 * PD;
      float* po = pooled + v0 * PD;
      int32_t* a = arg + v0 * PD;
      float* mx = mmax + v0 * PD;
      switch (V - v0 < 4 ? V - v0 : 4) {
        case 1: pool_drop_pairs_kernel<T, 1><<<blocks, 128, 0, s>>>((const T*)h, ldh, sent_ptr, pair_sent, pair_row_ptr, P, D, chunks, g, mv, po, a, mx); break;
        case 2: pool_drop_pairs_kernel<T, 2><<<blocks, 128, 0, s>>>((const T*)h, ldh, sent_ptr, pair_sent, pair_row_ptr, P, D, chunks, g, mv, po, a, mx); break;
        case 3: pool_drop_pairs_kernel<T, 3><<<blocks, 128, 0, s>>>((const T*)h, ldh, sent_ptr, pair_sent, pair_row_ptr, P, D, chunks, g, mv, po, a, mx); break;
        default: pool_drop_pairs_kernel<T, 4><<<blocks, 128, 0, s>>>((const T*)h, ldh, sent_ptr, pair_sent, pair_row_ptr, P, D, chunks, g, mv, po, a, mx); break;
      }
    }
  })
  return check_launch();
}

extern "C" int edg_views_bwd_drop_pairs(const float* pooled, const float* mmax, const int32_t* arg, const float* gates,
                                        const float* g_xy, int32_t V, const int32_t* sent_ptr, const int32_t* row_sent,
                                        int32_t N, const int32_t* pair_ptr, const int32_t* pair_row_ptr, int32_t P,
                                        int32_t D, const int64_t* seed, float p, void* dh, int dtype, int64_t lddh,
                                        float* dgates, int acc_view, edg_stream stream) {
  if (V <= 0 || N < 0 || P < 0 || D <= 0) return EDG_ERR_ARG;
  if (P == 0) return EDG_OK;
  if (!pooled || !gates || (!dh && !dgates)) return EDG_ERR_ARG;
  if (dgates && !mmax) return EDG_ERR_ARG;
  if (dh && (!arg || !sent_ptr || !pair_ptr || !pair_row_ptr || (N > 0 && !row_sent))) return EDG_ERR_ARG;
  if (dh && (!aligned16(dh) || !row_pitch_ok(dtype, lddh))) return EDG_ERR_ALIGN;
  GateDrop m;
  if (const int rc = gate_drop(seed, 0, p, nullptr, m)) return rc;
  cudaStream_t s = (cudaStream_t)stream;
  if (dgates) {
    const int64_t total = (int64_t)P * D;
    views_dgates_drop_pairs_kernel<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(pooled, mmax, g_xy, V, P, D, dgates,
                                                                                 acc_view);
  }
  if (dh && N > 0) {
    EDG_DISPATCH_T(dtype, {
      constexpr int E = Vec16<T>::kElems;
      const int chunks = (D + E - 1) / E;
      const unsigned blocks = (unsigned)(((int64_t)N * chunks + 127) / 128);
      views_dh_drop_pairs_kernel<T><<<blocks, 128, 0, s>>>(pooled, arg, gates, g_xy, V, sent_ptr, row_sent, pair_ptr,
                                                           pair_row_ptr, N, P, D, chunks, m, (T*)dh, lddh);
    })
  }
  return check_launch();
}

extern "C" int edg_views_bwd_hmax_pairs(const float* hmax, const float* gates, const float* g_xy, int32_t V, int32_t S,
                                        const int32_t* pair_ptr, int32_t P, int32_t D, float* patch_val, int64_t ldp,
                                        float* dgates, int acc_view, edg_stream stream) {
  if (V <= 0 || S < 0 || P < 0 || D <= 0 || ldp < D) return EDG_ERR_ARG;
  if (S == 0) return EDG_OK;
  if (!hmax || !pair_ptr || !patch_val || (P > 0 && (!gates || !dgates))) return EDG_ERR_ARG;
  const int64_t total = (int64_t)S * D;
  views_bwd_hmax_pairs_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
      hmax, gates, g_xy, V, S, pair_ptr, P, D, patch_val, ldp, dgates, acc_view);
  return check_launch();
}

extern "C" int edg_trigger_scatter_add_pairs(const float* da, const float* extra, int32_t n_extra, int32_t S,
                                             const int32_t* pair_ptr, int32_t P, int32_t D, const int32_t* pair_start,
                                             const int32_t* anchor, void* dx, int dtype, int64_t lddx, edg_stream stream) {
  if (S < 0 || P < 0 || D <= 0 || n_extra < 0) return EDG_ERR_ARG;
  if (S == 0 || P == 0) return EDG_OK;
  if ((!da && n_extra == 0) || (n_extra > 0 && !extra) || !pair_ptr || !pair_start || !anchor || !dx) return EDG_ERR_ARG;
  cudaStream_t s = (cudaStream_t)stream;
  EDG_DISPATCH_T(dtype, trigger_scatter_add_pairs_kernel<T><<<blocks_for((int64_t)S * D, 256), 256, 0, s>>>(
      da, extra, n_extra, S, pair_ptr, P, D, pair_start, anchor, (T*)dx, lddx);)
  return check_launch();
}
