// Every candidate trigger of a sentence from one pass of the GCN chain (include/edgcn.h, "Trigger pairs").
//
// The GCN chain h_1 .. h_L depends on the sentence and not on the trigger, so the rows of a sentence exist once, and
// only what depends on the trigger runs per (sentence, trigger) pair p: the scores / kl of bert_amir5.py:645-648 over
// the sentence's rows against that pair's g_p * v_p, and their backward.  The pairs of sentence s are the contiguous
// range pair_ptr[s] .. pair_ptr[s+1] - 1; per-pair row outputs (scores, dist, ...) live in the per-pair packed layout
// whose pair p starts at pair_row_ptr[p].  Every sum over the pairs of a sentence runs in ascending pair order inside
// one thread (no atomics), so the results do not depend on scheduling.
//
// Included after edg_block.cu (softmax_stats, dist_at, ScoresQ).

namespace edg {

// ---- scores, softmax product and d kl / d (v, c) units per pair -----------------------------------------
// One warp per pair (the per-pair twin of scores_kl_fwd_kernel): the sentence's rows are read through L1 / L2, where
// the consecutive pairs of a sentence -- consecutive warps of a block -- find them.
template <typename T, int I64>
__global__ void __launch_bounds__(128)
scores_kl_pairs_kernel(const T* __restrict__ h, int64_t ldh, const int32_t* __restrict__ sent_ptr,
                       const int32_t* __restrict__ pair_sent, const int32_t* __restrict__ pair_row_ptr, int P, int D,
                       int chunks, const float* __restrict__ gate, const float* __restrict__ vvec,
                       const float* __restrict__ cvec, const void* __restrict__ dist, float* __restrict__ scores,
                       float* __restrict__ kl_b, float* __restrict__ dv_unit, float* __restrict__ dc_unit,
                       float* __restrict__ u_unit, float* __restrict__ sf_unit) {
  constexpr int E = Vec16<T>::kElems;
  constexpr int kMaxQ = ScoresQ<T>::value;
  const int p = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (p >= P) return;
  const int lane = threadIdx.x & 31;
  const int s = __ldg(pair_sent + p);
  const int beg = __ldg(sent_ptr + s), end = __ldg(sent_ptr + s + 1), n = end - beg;
  const int o0 = __ldg(pair_row_ptr + p);                 // this pair's rows in the per-pair layout
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
template <typename T, int I64>
__global__ void __launch_bounds__(128)
head_pairs_kernel(const T* __restrict__ h, int64_t ldh, const int32_t* __restrict__ sent_ptr,
                  const int32_t* __restrict__ pair_sent, const int32_t* __restrict__ pair_row_ptr, int P, int D, int chunks,
                  const float* __restrict__ gate, const float* __restrict__ vvec, const void* __restrict__ dist,
                  const float* __restrict__ scores, const float* __restrict__ kl_b, const float* __restrict__ g_kl,
                  const float* __restrict__ g_scores, const float* __restrict__ g_pooled, const int32_t* __restrict__ arg,
                  float* __restrict__ ds_ws, float* __restrict__ dgate, float* __restrict__ dv, float* __restrict__ dc) {
  constexpr int E = Vec16<T>::kElems;
  constexpr int kMaxQ = ScoresQ<T>::value;
  const int p = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (p >= P) return;
  const int lane = threadIdx.x & 31;
  const int s = __ldg(pair_sent + p);
  const int beg = __ldg(sent_ptr + s), end = __ldg(sent_ptr + s + 1), n = end - beg;
  const int o0 = __ldg(pair_row_ptr + p);
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
            const int r = __ldg(arg + (int64_t)s * D + c + k);
            if (r >= beg && r < end) dg = fmaf(__ldg(g_pooled + o), to_f32(h[(int64_t)r * ldh + c + k]), dg);
          }
          dgate[o] = dg;
        }
      }
  }
}

// ---- head backward, row part: d h_L over the sentence rows ----------------------------------------------------
// thread = (row, 16-byte column chunk):  dh_t = sum_p ds_{p,t} (g_p v_p)  +  [t = arg_s] sum_p g_p g_pooled_p,
// the pairs of the row's sentence in ascending order.  Every row is written (0 where the sentence has no pairs).
template <typename T>
__global__ void __launch_bounds__(128)
dh_pairs_kernel(const int32_t* __restrict__ sent_ptr, const int32_t* __restrict__ row_sent,
                const int32_t* __restrict__ pair_ptr, const int32_t* __restrict__ pair_row_ptr, int N, int D, int chunks,
                const float* __restrict__ gate, const float* __restrict__ vvec, const float* __restrict__ g_pooled,
                const int32_t* __restrict__ arg, const float* __restrict__ ds_ws, int have_s, T* __restrict__ dh,
                int64_t lddh) {
  constexpr int E = Vec16<T>::kElems;
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int t = (int)(idx / chunks);
  if (t >= N) return;
  const int c = (int)(idx - (int64_t)t * chunks) * E;
  const int s = __ldg(row_sent + t);
  const int loc = t - __ldg(sent_ptr + s);
  const int p0 = __ldg(pair_ptr + s), p1 = __ldg(pair_ptr + s + 1);
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

extern "C" int edg_scores_kl_pairs_fwd(const void* h, int dtype, int64_t ldh, const int32_t* sent_ptr,
                                       const int32_t* pair_sent, const int32_t* pair_row_ptr, int32_t P, int32_t D,
                                       const float* gate, const float* v, const float* c, const void* dist, int dist_i64,
                                       float* scores, float* kl_b, float* dv_unit, float* dc_unit, float* u_unit,
                                       float* sf_unit, edg_stream stream) {
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
                                                          gate, v, c, dist, scores, kl_b, dv_unit, dc_unit, u_unit, sf_unit);
    else
      scores_kl_pairs_kernel<T, 0><<<blocks, 128, 0, s>>>((const T*)h, ldh, sent_ptr, pair_sent, pair_row_ptr, P, D, chunks,
                                                          gate, v, c, dist, scores, kl_b, dv_unit, dc_unit, u_unit, sf_unit);
  })
  return check_launch();
}

extern "C" int edg_head_bwd_pairs(const void* h, int dtype, int64_t ldh, const int32_t* sent_ptr, int32_t S,
                                  const int32_t* row_sent, int32_t N, const int32_t* pair_ptr, const int32_t* pair_sent, const int32_t* pair_row_ptr, int32_t P,
                                  int32_t D, const float* gate, const float* v, const void* dist, int dist_i64,
                                  const float* scores, const float* kl_b, const float* g_kl, const float* g_scores,
                                  const float* g_pooled, const int32_t* arg, void* dh, int64_t lddh, float* dgate,
                                  float* dv, float* dc, float* ds_ws, edg_stream stream) {
  if (S < 0 || P < 0 || D <= 0) return EDG_ERR_ARG;
  if (!sent_ptr || !pair_ptr || !pair_sent || !pair_row_ptr || !gate || !h || !ds_ws) return EDG_ERR_ARG;
  if (!dh && !dv && !dc) return EDG_ERR_ARG;
  if (dh && (!dgate || N < 0 || (N > 0 && !row_sent))) return EDG_ERR_ARG;
  if (g_pooled && !arg) return EDG_ERR_ARG;
  if ((g_kl || g_scores) && (!scores || !v)) return EDG_ERR_ARG;
  if (g_kl && (!dist || !kl_b)) return EDG_ERR_ARG;
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
                                                       v, dist, scores, kl_b, g_kl, g_scores, g_pooled, arg, ds_ws, dgate, dv, dc);
      else
        head_pairs_kernel<T, 0><<<blocks, 128, 0, s>>>((const T*)h, ldh, sent_ptr, pair_sent, pair_row_ptr, P, D, chunks, gate,
                                                       v, dist, scores, kl_b, g_kl, g_scores, g_pooled, arg, ds_ws, dgate, dv, dc);
    }
    if (dh && N > 0) {
      const unsigned blocks = (unsigned)(((int64_t)N * chunks + 127) / 128);
      dh_pairs_kernel<T><<<blocks, 128, 0, s>>>(sent_ptr, row_sent, pair_ptr, pair_row_ptr, N, D, chunks, gate, v, g_pooled,
                                                arg, ds_ws, have_s, (T*)dh, lddh);
    }
  })
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
