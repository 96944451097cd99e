// Kernels of the gated block around the graph convolution (models/bert_amir5.py:615-648):
// trigger gather, gated max-pool views, gate-diversity term, collapsed importance scores
// + softmax product ("kl"), and their backward passes.  All HBM/L2-bound row streaming:
// 128-bit loads along the hidden dimension, one pass over the [N,D] matrix per kernel.
#include <math.h>
#include <stdlib.h>

#include "edg_common.cuh"

namespace edg {

// ---- trigger row ------------------------------------------------------------
template <typename T>
__global__ void trigger_gather_kernel(const T* __restrict__ x, int64_t ldx, const int32_t* __restrict__ sent_ptr,
                                      const int32_t* __restrict__ anchor, int B, int D, float* __restrict__ raw,
                                      T* __restrict__ act, int64_t ldact, int lead_sigmoid) {
  // covers [B, ldact]: the padding columns of `act` are written as zeros
  const int W = act ? (int)ldact : D;
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int b = (int)(idx / W);
  if (b >= B) return;
  const int d = (int)(idx - (int64_t)b * W);
  if (d >= D) { act[(int64_t)b * ldact + d] = from_f32<T>(0.f); return; }
  const int64_t row = (int64_t)sent_ptr[b] + anchor[b];
  const float v = to_f32(x[row * ldx + d]);
  if (raw) raw[(int64_t)b * D + d] = v;
  if (act) act[(int64_t)b * ldact + d] = from_f32<T>(lead_sigmoid ? sigmoidf_(v) : v);
}

// da (optional) plus `n_extra` more [B, D] terms stored one after the other in `extra` (the gate MLPs' input gradients
// come as one [L, B, D] array): summed here instead of by separate elementwise launches
template <typename T>
__global__ void trigger_scatter_add_kernel(const float* __restrict__ da, const float* __restrict__ extra, int n_extra, int B,
                                           int D, const int32_t* __restrict__ sent_ptr, const int32_t* __restrict__ anchor,
                                           T* __restrict__ dx, int64_t lddx) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int b = (int)(idx / D);
  if (b >= B) return;
  const int d = (int)(idx - (int64_t)b * D);
  const int64_t row = (int64_t)sent_ptr[b] + anchor[b];
  T* p = dx + row * lddx + d;
  const int64_t e = (int64_t)b * D + d, BD = (int64_t)B * D;
  float v = da ? da[e] : 0.f;
  for (int k = 0; k < n_extra; ++k) v += extra[k * BD + e];
  *p = from_f32<T>(to_f32(*p) + v);
}

// ---- gated max-pool views ---------------------------------------------------
template <typename T, int V>
__global__ void __launch_bounds__(128)
pool_fwd_kernel(const T* __restrict__ h, int64_t ldh, const int32_t* __restrict__ sent_ptr, int B, int D, int chunks,
                const float* __restrict__ gates, float* __restrict__ pooled, int32_t* __restrict__ arg,
                float* __restrict__ hmax) {
  // same rule as pool_staged_kernel: gate-independent column maximum + first row, one multiply per view
  constexpr int E = Vec16<T>::kElems;
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int b = (int)(idx / chunks);
  if (b >= B) return;
  const int c = (int)(idx - (int64_t)b * chunks) * E;
  const int64_t BD = (int64_t)B * D;
  const int beg = sent_ptr[b], end = sent_ptr[b + 1];
  float m[E];
  int32_t where[E];
#pragma unroll
  for (int k = 0; k < E; ++k) { m[k] = -INFINITY; where[k] = beg; }
  constexpr int U = 4;                        // rows in flight per thread (memory-level parallelism)
  for (int t = beg; t < end; t += U) {
    float f[U][E];
#pragma unroll
    for (int u = 0; u < U; ++u)
      if (t + u < end) Vec16<T>::load(h + (int64_t)(t + u) * ldh + c, f[u]);
#pragma unroll
    for (int u = 0; u < U; ++u) {
      if (t + u >= end) break;
#pragma unroll
      for (int k = 0; k < E; ++k)
        if (f[u][k] > m[k]) { m[k] = f[u][k]; where[k] = t + u; }       // strict: first row wins ties
    }
  }
#pragma unroll
  for (int v = 0; v < V; ++v)
#pragma unroll
    for (int k = 0; k < E; ++k)
      if (c + k < D) {
        const float g = __ldg(gates + v * BD + (int64_t)b * D + c + k);
        const int64_t o = v * BD + (int64_t)b * D + c + k;
        pooled[o] = (beg < end) ? m[k] * g : 0.f;
        arg[o] = (beg < end) ? (g != 0.f ? where[k] : beg) : -1;
      }
  if (hmax)
#pragma unroll
    for (int k = 0; k < E; ++k)
      if (c + k < D) hmax[(int64_t)b * D + c + k] = (beg < end) ? m[k] : 0.f;
}

// ---- diversity term -----------------------------------------------------------
__global__ void __launch_bounds__(256)
diversity_partial_kernel(const float* __restrict__ pooled, int V, int64_t BD, float* __restrict__ partial) {
  __shared__ float red[8];
  float s = 0.f;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < BD; i += (int64_t)gridDim.x * blockDim.x) {
    for (int v = 0; v < V; ++v) {
      const float pv = pooled[v * BD + i];
      for (int u = v + 1; u < V; ++u) s = fmaf(pv, pooled[u * BD + i], s);
    }
  }
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int w = 0; w < 8; ++w) t += red[w];
    partial[blockIdx.x] = t;
  }
}

// out = scale * sum(in[0..n)) in a fixed order, double accumulation
__global__ void __launch_bounds__(256)
sum_scaled_kernel(const float* __restrict__ in, int64_t n, float scale, float* __restrict__ out) {
  __shared__ double red[256];
  double s = 0.0;
  for (int64_t i = threadIdx.x; i < n; i += 256) s += (double)in[i];
  red[threadIdx.x] = s;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) out[0] = (float)(red[0] * (double)scale);
}

// ---- backward of the views + diversity ------------------------------------------
// parts: bit 0 = add the views' gradient into dh (scattered read-modify-write), bit 1 = dgates (gathers h at the
// arg-max rows).  The two halves have different consumers (layer 1's backward / the gate MLPs' backward), so the
// caller may issue them as two launches on two streams.
// latency-bound scattered gathers / read-modify-writes: occupancy is what helps.  Uncapped the kernel takes 80 registers
// (3 blocks per SM, 68 us at C2); capped to 32 registers for 8 resident blocks it runs in 48 us (104 bytes of spills),
// same-box A/B of the whole step 0.915 vs 0.953 ms
#ifndef EDG_VIEWS_MINBLOCKS
#define EDG_VIEWS_MINBLOCKS 8
#endif
template <typename T>
__global__ void __launch_bounds__(256, EDG_VIEWS_MINBLOCKS)
views_bwd_kernel(const float* __restrict__ pooled, const int32_t* __restrict__ arg, const float* __restrict__ gates,
                 const T* __restrict__ h, int64_t ldh, int V, int B, int D, const float* __restrict__ g_xy,
                 const float* __restrict__ g_pooled, T* __restrict__ dh, int64_t lddh, float* __restrict__ dgates,
                 int acc_view, int parts) {
  const int64_t BD = (int64_t)B * D;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= BD) return;
  const int d = (int)(i % D);
  const float gxy = g_xy ? (__ldg(g_xy) / (float)B) : 0.f;
  float tot = 0.f;
  for (int v = 0; v < V; ++v) tot += pooled[v * BD + i];
  for (int v = 0; v < V; ++v) {
    float dp = gxy * (tot - pooled[v * BD + i]);
    if (g_pooled) dp += g_pooled[v * BD + i];
    const int r = arg[v * BD + i];
    float dgv = 0.f;
    if (r >= 0) {
      if (parts & 2) dgv = dp * to_f32(h[(int64_t)r * ldh + d]);
      if (parts & 1) {
        T* p = dh + (int64_t)r * lddh + d;                 // this thread owns column d of sentence b
        *p = from_f32<T>(to_f32(*p) + dp * gates[v * BD + i]);
      }
    }
    if (parts & 2) dgates[v * BD + i] = (v == acc_view) ? dgates[v * BD + i] + dgv : dgv;    // acc_view already holds d gate_L
  }
}

// ---- importance scores + softmax product ("kl") ---------------------------------
template <int I64> __device__ __forceinline__ float dist_at(const void* dist, int64_t i) {
  return I64 ? (float)reinterpret_cast<const long long*>(dist)[i] : (float)reinterpret_cast<const int32_t*>(dist)[i];
}

// softmax statistics of scores and of float(dist) over rows [beg,end) -- whole warp
template <int I64>
__device__ __forceinline__ void softmax_stats(const float* scores, const void* dist, int beg, int end, int lane,
                                              float& ms, float& zs, float& mq, float& zq) {
  ms = -INFINITY; mq = -INFINITY;
  for (int t = beg + lane; t < end; t += 32) {
    ms = fmaxf(ms, scores[t]);
    mq = fmaxf(mq, dist_at<I64>(dist, t));
  }
  ms = warp_max(ms); mq = warp_max(mq);
  zs = 0.f; zq = 0.f;
  for (int t = beg + lane; t < end; t += 32) {
    zs += expf(scores[t] - ms);
    zq += expf(dist_at<I64>(dist, t) - mq);
  }
  zs = warp_sum(zs); zq = warp_sum(zq);
}

// 16-byte chunks per lane: 32 fp32 values per lane either way, i.e. D <= 1024 for both dtypes
template <typename T> struct ScoresQ { static constexpr int value = 32 / Vec16<T>::kElems; };

template <typename T, int I64>
__global__ void __launch_bounds__(128)
scores_kl_fwd_kernel(const T* __restrict__ h, int64_t ldh, const int32_t* __restrict__ sent_ptr, int B, int D,
                     int chunks, const float* __restrict__ gate, const float* __restrict__ vvec,
                     const float* __restrict__ cvec, const void* __restrict__ dist, float* __restrict__ scores,
                     float* __restrict__ kl_b, float* __restrict__ dv_unit, float* __restrict__ dc_unit,
                     float* __restrict__ u_unit, float* __restrict__ sf_unit) {
  constexpr int E = Vec16<T>::kElems;
  constexpr int kMaxQ = ScoresQ<T>::value;
  const int b = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (b >= B) return;
  const int lane = threadIdx.x & 31;
  const int beg = sent_ptr[b], end = sent_ptr[b + 1];
  float w[kMaxQ][E];
#pragma unroll
  for (int q = 0; q < kMaxQ; ++q) {
    const int c = (lane + 32 * q) * E;
#pragma unroll
    for (int k = 0; k < E; ++k)
      w[q][k] = (lane + 32 * q < chunks && c + k < D)
                    ? __ldg(gate + (int64_t)b * D + c + k) * __ldg(vvec + (int64_t)b * D + c + k) : 0.f;
  }
  const float cb = cvec ? __ldg(cvec + b) : 0.f;
  constexpr int U = 4;                        // rows in flight per warp
  for (int t = beg; t < end; t += U) {
    float sacc[U];
#pragma unroll
    for (int u = 0; u < U; ++u) sacc[u] = 0.f;
#pragma unroll
    for (int q = 0; q < kMaxQ; ++q) {
      if (lane + 32 * q < chunks) {
        float f[U][E];
#pragma unroll
        for (int u = 0; u < U; ++u)
          if (t + u < end) Vec16<T>::load(h + (int64_t)(t + u) * ldh + (lane + 32 * q) * E, f[u]);
#pragma unroll
        for (int u = 0; u < U; ++u)
          if (t + u < end) {
#pragma unroll
            for (int k = 0; k < E; ++k) sacc[u] = fmaf(f[u][k], w[q][k], sacc[u]);
          }
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) sacc[u] = warp_sum(sacc[u]);
    if (lane < U && t + lane < end) {
      float mine = sacc[0];
#pragma unroll
      for (int u = 1; u < U; ++u) mine = (lane == u) ? sacc[u] : mine;
      scores[t + lane] = mine + cb;
    }
  }
  __syncwarp();
  float ms, zs, mq, zq;
  softmax_stats<I64>(scores, dist, beg, end, lane, ms, zs, mq, zq);
  float acc = 0.f;
  for (int t = beg + lane; t < end; t += 32)
    acc += (expf(scores[t] - ms) / zs) * (expf(dist_at<I64>(dist, t) - mq) / zq);
  acc = warp_sum(acc);
  if (lane == 0) kl_b[b] = acc;
  if (dv_unit == nullptr) return;
  // d kl / d v_b and d kl / d c_b per unit upstream gradient (the backward pass only scales them):
  //   u_t = P_t (Q_t - kl_b) / B,  dv_unit[d] = sum_t u_t h[t,d] gate[d],  dc_unit = sum_t u_t
  // second sweep over the sentence's rows (just read: L1/L2 hits)
  const float klb = acc, invB = 1.0f / (float)B;
  float dvu[kMaxQ][E];
#pragma unroll
  for (int q = 0; q < kMaxQ; ++q)
#pragma unroll
    for (int k = 0; k < E; ++k) dvu[q][k] = 0.f;
  float dcu = 0.f;
  for (int t = beg; t < end; ++t) {
    const float u = (expf(scores[t] - ms) / zs) * ((expf(dist_at<I64>(dist, t) - mq) / zq) - klb) * invB;
    dcu += u;
    if (lane == 0 && u_unit) u_unit[t] = u;
#pragma unroll
    for (int q = 0; q < kMaxQ; ++q) {
      if (lane + 32 * q < chunks) {
        float f[E];
        Vec16<T>::load(h + (int64_t)t * ldh + (lane + 32 * q) * E, f);
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
      if (lane + 32 * q < chunks && c + k < D)
      {
        dv_unit[(int64_t)b * D + c + k] = dvu[q][k] * __ldg(gate + (int64_t)b * D + c + k);
        if (sf_unit) sf_unit[(int64_t)b * D + c + k] = dvu[q][k];
      }
  }
  if (lane == 0 && dc_unit) dc_unit[b] = dcu;
}

// one block per sentence; phase 1: ds[t] into shared memory; phase 2: thread = 16-byte
// column chunk, streaming the sentence's rows once.
template <typename T, int I64>
__global__ void __launch_bounds__(256)
head_bwd_kernel(const T* __restrict__ h, int64_t ldh, const int32_t* __restrict__ sent_ptr, int B, int D, int chunks,
                const float* __restrict__ gate, const float* __restrict__ vvec, const void* __restrict__ dist,
                const float* __restrict__ scores, const float* __restrict__ kl_b, const float* __restrict__ g_kl,
                const float* __restrict__ g_scores, const float* __restrict__ g_pooled, const int32_t* __restrict__ arg,
                const T* __restrict__ g_xout, int64_t ldgx, T* __restrict__ dh, int64_t lddh,
                float* __restrict__ dgate, float* __restrict__ dv, float* __restrict__ dc) {
  constexpr int E = Vec16<T>::kElems;
  extern __shared__ float ds[];
  const int b = blockIdx.x;
  const int beg = sent_ptr[b], end = sent_ptr[b + 1], n = end - beg;
  const bool have_s = (scores != nullptr) && (g_kl != nullptr || g_scores != nullptr);
  if (threadIdx.x < 32) {
    const int lane = threadIdx.x;
    if (have_s) {
      float ms = 0.f, zs = 1.f, mq = 0.f, zq = 1.f;
      const float gk = g_kl ? (__ldg(g_kl) / (float)B) : 0.f;
      if (g_kl) softmax_stats<I64>(scores, dist, beg, end, lane, ms, zs, mq, zq);
      const float klb = g_kl ? kl_b[b] : 0.f;
      float tot = 0.f;
      for (int t = beg + lane; t < end; t += 32) {
        float v = 0.f;
        if (g_kl) {
          const float P = expf(scores[t] - ms) / zs, Q = expf(dist_at<I64>(dist, t) - mq) / zq;
          v = gk * P * (Q - klb);
        }
        if (g_scores) v += g_scores[t];
        ds[t - beg] = v;
        tot += v;
      }
      tot = warp_sum(tot);
      if (lane == 0 && dc) dc[b] = tot;
    } else {
      for (int t = lane; t < n; t += 32) ds[t] = 0.f;
      if (lane == 0 && dc) dc[b] = 0.f;
    }
  }
  __syncthreads();
  if ((int)threadIdx.x >= chunks) return;
  const int c = threadIdx.x * E;
  float g[E], vv[E], gp[E], ag[E], av[E];
  int32_t where[E];
#pragma unroll
  for (int k = 0; k < E; ++k) {
    const bool ok = c + k < D;
    const int64_t o = (int64_t)b * D + c + k;
    g[k] = ok ? __ldg(gate + o) : 0.f;
    vv[k] = (ok && vvec) ? __ldg(vvec + o) : 0.f;
    gp[k] = (ok && g_pooled) ? __ldg(g_pooled + o) : 0.f;
    where[k] = (ok && g_pooled) ? __ldg(arg + o) : -1;
    ag[k] = 0.f; av[k] = 0.f;
  }
  constexpr int U = 4;                        // rows in flight per thread
  for (int t0 = beg; t0 < end; t0 += U) {
    float f[U][E], gx[U][E];
#pragma unroll
    for (int u = 0; u < U; ++u)
      if (t0 + u < end) {
        Vec16<T>::load(h + (int64_t)(t0 + u) * ldh + c, f[u]);
        if (g_xout) Vec16<T>::load(g_xout + (int64_t)(t0 + u) * ldgx + c, gx[u]);
      }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int t = t0 + u;
      if (t >= end) break;
      float o[E];
      const float dst = ds[t - beg];
#pragma unroll
      for (int k = 0; k < E; ++k) {
        float coef = dst * vv[k];
        if (where[k] == t) coef += gp[k];
        if (g_xout) coef += gx[u][k];
        o[k] = g[k] * coef;
        ag[k] = fmaf(f[u][k], coef, ag[k]);
        av[k] = fmaf(dst * f[u][k], g[k], av[k]);
      }
      if (dh) Vec16<T>::store(dh + (int64_t)t * lddh + c, o);
    }
  }
#pragma unroll
  for (int k = 0; k < E; ++k)
    if (c + k < D) {
      const int64_t o = (int64_t)b * D + c + k;
      if (dgate) dgate[o] = ag[k];
      if (dv) dv[o] = av[k];
    }
}

template <typename T, typename TO>
__global__ void __launch_bounds__(128)
gate_rows_kernel(const T* __restrict__ h, int64_t ldh, const int32_t* __restrict__ sent_ptr, int B, int D, int chunks,
                 const float* __restrict__ gate, TO* __restrict__ out, int64_t ldo, int act) {
  constexpr int E = Vec16<T>::kElems;
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int b = (int)(idx / chunks);
  if (b >= B) return;
  const int c = (int)(idx - (int64_t)b * chunks) * E;
  float g[E];
#pragma unroll
  for (int k = 0; k < E; ++k) g[k] = (c + k < D) ? __ldg(gate + (int64_t)b * D + c + k) : 0.f;
  for (int t = sent_ptr[b]; t < sent_ptr[b + 1]; ++t) {
    float f[E];
    Vec16<T>::load(h + (int64_t)t * ldh + c, f);
#pragma unroll
    for (int k = 0; k < E; ++k)
      if (c + k < D) {
        const float v = f[k] * g[k];
        out[(int64_t)t * ldo + c + k] = from_f32<TO>(act == EDG_ACT_SIGMOID ? sigmoidf_(v) : v);
      }
  }
}

__global__ void sigmoid_bwd_kernel(const void* __restrict__ y, int y_dtype, int64_t ldy, const void* __restrict__ dy,
                                   int dy_dtype, int64_t lddy, int R, int C, void* __restrict__ dz, int dz_dtype,
                                   int64_t lddz, int accumulate) {
  // covers the whole [R, lddz] allocation: padding columns are written as zeros (no separate memset)
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int W = (int)lddz;
  const int r = (int)(idx / W);
  if (r >= R) return;
  const int c = (int)(idx - (int64_t)r * W);
  float v = 0.f;
  if (c < C) {
    const float yv = load_as_f32(y, y_dtype, (int64_t)r * ldy + c);
    v = load_as_f32(dy, dy_dtype, (int64_t)r * lddy + c) * yv * (1.f - yv);
    if (accumulate) v += load_as_f32(dz, dz_dtype, (int64_t)r * lddz + c);
  }
  store_from_f32(dz, dz_dtype, (int64_t)r * lddz + c, v);
}

__global__ void cast_2d_kernel(const float* __restrict__ src, int64_t lds, int R, int C, void* __restrict__ dst,
                               int dst_dtype, int64_t ldd, int transpose) {
  const int rows_out = transpose ? C : R, cols_out = transpose ? R : C;
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int ro = (int)(idx / ldd);
  if (ro >= rows_out) return;
  const int co = (int)(idx - (int64_t)ro * ldd);
  float v = 0.f;
  if (co < cols_out) v = transpose ? src[(int64_t)co * lds + ro] : src[(int64_t)ro * lds + co];
  store_from_f32(dst, dst_dtype, (int64_t)ro * ldd + co, v);
}

// all weight copies of a step in ONE launch: entry = blockIdx.y
constexpr int kCastBatchMax = 32;
struct CastBatch {
  const float* src[kCastBatchMax];
  void* dst[kCastBatchMax];
  int R[kCastBatchMax], C[kCastBatchMax], lds[kCastBatchMax], ldd[kCastBatchMax], transpose[kCastBatchMax];
};
__global__ void cast_batch_kernel(const __grid_constant__ CastBatch b, int dst_dtype) {
  const int e = blockIdx.y;
  const int R = b.R[e], C = b.C[e], ldd = b.ldd[e], tr = b.transpose[e];
  const int rows_out = tr ? C : R, cols_out = tr ? R : C;
  const float* __restrict__ src = b.src[e];
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < (int64_t)rows_out * ldd;
       idx += (int64_t)gridDim.x * blockDim.x) {
    const int ro = (int)(idx / ldd), co = (int)(idx - (int64_t)ro * ldd);
    float v = 0.f;
    if (co < cols_out) v = tr ? src[(int64_t)co * b.lds[e] + ro] : src[(int64_t)ro * b.lds[e] + co];
    store_from_f32(b.dst[e], dst_dtype, idx, v);
  }
}

}  // namespace edg

namespace edg {
template <typename T>
int pool_fwd_staged(const void* h, int64_t ldh, const int32_t* sent_ptr, const int32_t* row_sent, int N, int B, int D,
                    int max_len, const float* gates, int V, float* pooled, int32_t* arg, float* hmax, cudaStream_t s);
template <typename T>
int scores_kl_staged(const void* h, int64_t ldh, const int32_t* sent_ptr, const int32_t* row_sent, int N, int B, int D,
                     int max_len, const float* gate, const float* v, const float* c, const void* dist, int dist_i64,
                     float* scores, float* kl_b, float* dv_unit, float* dc_unit, float* u_unit, float* sf_unit, cudaStream_t s);
template <typename T>
int head_bwd_staged(const void* h, int64_t ldh, const int32_t* sent_ptr, const int32_t* row_sent, int N, int B, int D,
                    int max_len, const float* gate, const float* v, const void* dist, int dist_i64, const float* scores,
                    const float* kl_b, const float* g_kl, const float* g_scores, const float* g_pooled, const int32_t* arg,
                    const void* g_xout, int64_t ldgx, void* dh, int64_t lddh, float* dgate, float* dv, float* dc,
                    cudaStream_t s);
}  // namespace edg

using namespace edg;

#define EDG_DISPATCH_T(dtype, ...)                                \
  if ((dtype) == EDG_BF16) { using T = __nv_bfloat16; __VA_ARGS__ } \
  else if ((dtype) == EDG_F32) { using T = float; __VA_ARGS__ }     \
  else return EDG_ERR_DTYPE;

static inline unsigned blocks_for(int64_t total, int threads) { return (unsigned)((total + threads - 1) / threads); }

extern "C" int edg_trigger_gather(const void* x, int dtype, int64_t ldx, const int32_t* sent_ptr,
                                  const int32_t* anchor, int32_t B, int32_t D, float* raw, void* act,
                                  int64_t ldact, int lead_sigmoid, edg_stream stream) {
  if (B < 0 || D <= 0) return EDG_ERR_ARG;
  if (B == 0) return EDG_OK;
  if (!x || !sent_ptr || !anchor) return EDG_ERR_ARG;
  cudaStream_t s = (cudaStream_t)stream;
  EDG_DISPATCH_T(dtype, trigger_gather_kernel<T><<<blocks_for((int64_t)B * (act ? ldact : D), 256), 256, 0, s>>>(
      (const T*)x, ldx, sent_ptr, anchor, B, D, raw, (T*)act, ldact, lead_sigmoid);)
  return check_launch();
}

extern "C" int edg_trigger_scatter_add(const float* da, const float* extra, int32_t n_extra, int32_t B, int32_t D,
                                       const int32_t* sent_ptr, const int32_t* anchor, void* dx, int dtype, int64_t lddx,
                                       edg_stream stream) {
  if (B < 0 || D <= 0 || n_extra < 0) return EDG_ERR_ARG;
  if (B == 0) return EDG_OK;
  if ((!da && n_extra == 0) || (n_extra > 0 && !extra) || !sent_ptr || !anchor || !dx) return EDG_ERR_ARG;
  cudaStream_t s = (cudaStream_t)stream;
  EDG_DISPATCH_T(dtype, trigger_scatter_add_kernel<T><<<blocks_for((int64_t)B * D, 256), 256, 0, s>>>(
      da, extra, n_extra, B, D, sent_ptr, anchor, (T*)dx, lddx);)
  return check_launch();
}

template <typename T>
static int pool_fwd_dispatch(const void* h, int64_t ldh, const int32_t* sent_ptr, int B, int D, const float* gates,
                             int V, float* pooled, int32_t* arg, float* hmax, cudaStream_t s) {
  constexpr int E = Vec16<T>::kElems;
  const int chunks = (D + E - 1) / E;
  const unsigned blocks = blocks_for((int64_t)B * chunks, 128);
  const int64_t BD = (int64_t)B * D;
  for (int v0 = 0; v0 < V; v0 += 4) {
    const int nv = (V - v0) < 4 ? (V - v0) : 4;
    const float* g = gates + v0 * BD;
    float* p = pooled + v0 * BD;
    int32_t* a = arg + v0 * BD;
    switch (nv) {
      case 1: pool_fwd_kernel<T, 1><<<blocks, 128, 0, s>>>((const T*)h, ldh, sent_ptr, B, D, chunks, g, p, a, v0 == 0 ? hmax : nullptr); break;
      case 2: pool_fwd_kernel<T, 2><<<blocks, 128, 0, s>>>((const T*)h, ldh, sent_ptr, B, D, chunks, g, p, a, v0 == 0 ? hmax : nullptr); break;
      case 3: pool_fwd_kernel<T, 3><<<blocks, 128, 0, s>>>((const T*)h, ldh, sent_ptr, B, D, chunks, g, p, a, v0 == 0 ? hmax : nullptr); break;
      default: pool_fwd_kernel<T, 4><<<blocks, 128, 0, s>>>((const T*)h, ldh, sent_ptr, B, D, chunks, g, p, a, v0 == 0 ? hmax : nullptr); break;
    }
  }
  return check_launch();
}

extern "C" int edg_pool_fwd(const void* h, int dtype, int64_t ldh, const int32_t* sent_ptr, int32_t B,
                            int32_t D, const float* gates, int32_t V, float* pooled, int32_t* arg,
                            const int32_t* row_sent, int32_t N, int32_t max_len, float* hmax, edg_stream stream) {
  if (B < 0 || D <= 0 || V <= 0) return EDG_ERR_ARG;
  if (B == 0) return EDG_OK;
  if (!h || !sent_ptr || !gates || !pooled || !arg) return EDG_ERR_ARG;
  if (!aligned16(h) || !row_pitch_ok(dtype, ldh)) return EDG_ERR_ALIGN;
  cudaStream_t s = (cudaStream_t)stream;
  EDG_DISPATCH_T(dtype, {
    const int rc = pool_fwd_staged<T>(h, ldh, sent_ptr, row_sent, N, B, D, max_len, gates, V, pooled, arg, hmax, s);
    if (rc <= 0) return rc;
    return pool_fwd_dispatch<T>(h, ldh, sent_ptr, B, D, gates, V, pooled, arg, hmax, s);
  })
}

extern "C" int edg_sum_scaled(const float* in, int64_t n, float scale, float* out, edg_stream stream) {
  if (n < 0 || !out || (n > 0 && !in)) return EDG_ERR_ARG;
  sum_scaled_kernel<<<1, 256, 0, (cudaStream_t)stream>>>(in, n, scale, out);
  return check_launch();
}

extern "C" int edg_diversity_fwd(const float* pooled, int32_t V, int32_t B, int32_t D, float* xy, float* ws,
                                 edg_stream stream) {
  if (V <= 0 || B <= 0 || D <= 0 || !pooled || !xy || !ws) return EDG_ERR_ARG;
  cudaStream_t s = (cudaStream_t)stream;
  const int64_t BD = (int64_t)B * D;
  int blocks = (int)((BD + 255) / 256);
  if (blocks > 1024) blocks = 1024;
  diversity_partial_kernel<<<blocks, 256, 0, s>>>(pooled, V, BD, ws);
  sum_scaled_kernel<<<1, 256, 0, s>>>(ws, blocks, 1.0f / (float)B, xy);
  return check_launch();
}

static int views_bwd_entry(const float* pooled, const int32_t* arg, const float* gates, const void* h,
                           int dtype, int64_t ldh, int32_t V, int32_t B, int32_t D, const float* g_xy,
                           const float* g_pooled, void* dh, int64_t lddh, float* dgates, int acc_view, int parts,
                           edg_stream stream) {
  if (V <= 0 || B < 0 || D <= 0 || parts < 1 || parts > 3) return EDG_ERR_ARG;
  if (B == 0) return EDG_OK;
  if (!pooled || !arg || !gates) return EDG_ERR_ARG;
  if ((parts & 1) && !dh) return EDG_ERR_ARG;
  if ((parts & 2) && (!h || !dgates)) return EDG_ERR_ARG;
  cudaStream_t s = (cudaStream_t)stream;
  EDG_DISPATCH_T(dtype, views_bwd_kernel<T><<<blocks_for((int64_t)B * D, 256), 256, 0, s>>>(
      pooled, arg, gates, (const T*)h, ldh, V, B, D, g_xy, g_pooled, (T*)dh, lddh, dgates, acc_view, parts);)
  return check_launch();
}

extern "C" int edg_views_bwd(const float* pooled, const int32_t* arg, const float* gates, const void* h,
                             int dtype, int64_t ldh, int32_t V, int32_t B, int32_t D, const float* g_xy,
                             const float* g_pooled, void* dh, int64_t lddh, float* dgates, int acc_view,
                             edg_stream stream) {
  return views_bwd_entry(pooled, arg, gates, h, dtype, ldh, V, B, D, g_xy, g_pooled, dh, lddh, dgates, acc_view, 3, stream);
}

extern "C" int edg_views_bwd_parts(const float* pooled, const int32_t* arg, const float* gates, const void* h,
                                   int dtype, int64_t ldh, int32_t V, int32_t B, int32_t D, const float* g_xy,
                                   const float* g_pooled, void* dh, int64_t lddh, float* dgates, int acc_view,
                                   int parts, edg_stream stream) {
  return views_bwd_entry(pooled, arg, gates, h, dtype, ldh, V, B, D, g_xy, g_pooled, dh, lddh, dgates, acc_view, parts,
                         stream);
}

extern "C" int edg_scores_kl_fwd(const void* h, int dtype, int64_t ldh, const int32_t* sent_ptr, int32_t B,
                                 int32_t D, const float* gate, const float* v, const float* c,
                                 const void* dist, int dist_i64, float* scores, float* kl_b,
                                 float* dv_unit, float* dc_unit, float* u_unit, float* sf_unit,
                                 const int32_t* row_sent, int32_t N, int32_t max_len, edg_stream stream) {
  if (B < 0 || D <= 0) return EDG_ERR_ARG;
  if (B == 0) return EDG_OK;
  if (!h || !sent_ptr || !gate || !v || !dist || !scores || !kl_b) return EDG_ERR_ARG;
  if ((u_unit || sf_unit) && !dv_unit) return EDG_ERR_ARG;
  if (!aligned16(h) || !row_pitch_ok(dtype, ldh)) return EDG_ERR_ALIGN;
  cudaStream_t s = (cudaStream_t)stream;
  const unsigned blocks = blocks_for(B, 4);
  EDG_DISPATCH_T(dtype, {
    constexpr int E = Vec16<T>::kElems;
    const int chunks = (D + E - 1) / E;
    if (chunks > 32 * ScoresQ<T>::value) return EDG_ERR_UNSUPPORTED;
    const int rc = scores_kl_staged<T>(h, ldh, sent_ptr, row_sent, N, B, D, max_len, gate, v, c, dist, dist_i64, scores, kl_b,
                                       dv_unit, dc_unit, u_unit, sf_unit, s);
    if (rc <= 0) return rc;
    if (dist_i64) scores_kl_fwd_kernel<T, 1><<<blocks, 128, 0, s>>>((const T*)h, ldh, sent_ptr, B, D, chunks, gate, v, c, dist, scores, kl_b, dv_unit, dc_unit, u_unit, sf_unit);
    else scores_kl_fwd_kernel<T, 0><<<blocks, 128, 0, s>>>((const T*)h, ldh, sent_ptr, B, D, chunks, gate, v, c, dist, scores, kl_b, dv_unit, dc_unit, u_unit, sf_unit);
  })
  return check_launch();
}

extern "C" int edg_head_bwd(const void* h, int dtype, int64_t ldh, const int32_t* sent_ptr, int32_t B,
                            int32_t D, const float* gate, const float* v, const void* dist, int dist_i64,
                            const float* scores, const float* kl_b, const float* g_kl, const float* g_scores,
                            const float* g_pooled, const int32_t* arg, const void* g_xout, int64_t ldgx,
                            void* dh, int64_t lddh, float* dgate, float* dv, float* dc, int32_t max_len,
                            const int32_t* row_sent, int32_t N, edg_stream stream) {
  if (B < 0 || D <= 0 || max_len < 0) return EDG_ERR_ARG;
  if (B == 0) return EDG_OK;
  if (!h || !sent_ptr || !gate) return EDG_ERR_ARG;
  if (!dh && !dv) return EDG_ERR_ARG;
  if (g_pooled && !arg) return EDG_ERR_ARG;
  if ((g_kl || g_scores) && (!scores || !v)) return EDG_ERR_ARG;
  if (g_kl && (!dist || !kl_b)) return EDG_ERR_ARG;
  if (!aligned16(h) || !row_pitch_ok(dtype, ldh)) return EDG_ERR_ALIGN;
  if (dh && (!aligned16(dh) || !row_pitch_ok(dtype, lddh))) return EDG_ERR_ALIGN;
  if (g_xout && (!aligned16(g_xout) || !row_pitch_ok(dtype, ldgx))) return EDG_ERR_ALIGN;
  if (max_len > 8192) return EDG_ERR_UNSUPPORTED;
  cudaStream_t s = (cudaStream_t)stream;
  const size_t smem = (size_t)(max_len > 0 ? max_len : 1) * sizeof(float);
  EDG_DISPATCH_T(dtype, {
    constexpr int E = Vec16<T>::kElems;
    const int chunks = (D + E - 1) / E;
    if (chunks > 256) return EDG_ERR_UNSUPPORTED;
    const int rc = head_bwd_staged<T>(h, ldh, sent_ptr, row_sent, N, B, D, max_len, gate, v, dist, dist_i64, scores, kl_b, g_kl,
                                      g_scores, g_pooled, arg, g_xout, ldgx, dh, lddh, dgate, dv, dc, s);
    if (rc <= 0) return rc;
    int threads = ((chunks + 31) / 32) * 32;
    if (threads < 32) threads = 32;
    if (dist_i64) head_bwd_kernel<T, 1><<<B, threads, smem, s>>>((const T*)h, ldh, sent_ptr, B, D, chunks, gate, v, dist, scores, kl_b, g_kl, g_scores, g_pooled, arg, (const T*)g_xout, ldgx, (T*)dh, lddh, dgate, dv, dc);
    else head_bwd_kernel<T, 0><<<B, threads, smem, s>>>((const T*)h, ldh, sent_ptr, B, D, chunks, gate, v, dist, scores, kl_b, g_kl, g_scores, g_pooled, arg, (const T*)g_xout, ldgx, (T*)dh, lddh, dgate, dv, dc);
  })
  return check_launch();
}

static int gate_rows_entry(const void* h, int dtype, int64_t ldh, const int32_t* sent_ptr, int32_t B,
                           int32_t D, const float* gate, void* out, int out_dtype, int64_t ldo, int act,
                           edg_stream stream) {
  if (B < 0 || D <= 0 || (act != EDG_ACT_NONE && act != EDG_ACT_SIGMOID)) return EDG_ERR_ARG;
  if (B == 0) return EDG_OK;
  if (!h || !sent_ptr || !gate || !out) return EDG_ERR_ARG;
  if (!aligned16(h) || !row_pitch_ok(dtype, ldh)) return EDG_ERR_ALIGN;
  cudaStream_t s = (cudaStream_t)stream;
  EDG_DISPATCH_T(dtype, {
    constexpr int E = Vec16<T>::kElems;
    const int chunks = (D + E - 1) / E;
    const unsigned blocks = blocks_for((int64_t)B * chunks, 128);
    if (out_dtype == EDG_F32) gate_rows_kernel<T, float><<<blocks, 128, 0, s>>>((const T*)h, ldh, sent_ptr, B, D, chunks, gate, (float*)out, ldo, act);
    else if (out_dtype == EDG_BF16) gate_rows_kernel<T, __nv_bfloat16><<<blocks, 128, 0, s>>>((const T*)h, ldh, sent_ptr, B, D, chunks, gate, (__nv_bfloat16*)out, ldo, act);
    else return EDG_ERR_DTYPE;
  })
  return check_launch();
}

extern "C" int edg_gate_rows(const void* h, int dtype, int64_t ldh, const int32_t* sent_ptr, int32_t B,
                             int32_t D, const float* gate, void* out, int out_dtype, int64_t ldo,
                             edg_stream stream) {
  return gate_rows_entry(h, dtype, ldh, sent_ptr, B, D, gate, out, out_dtype, ldo, EDG_ACT_NONE, stream);
}

extern "C" int edg_gate_rows_act(const void* h, int dtype, int64_t ldh, const int32_t* sent_ptr, int32_t B,
                                 int32_t D, const float* gate, void* out, int out_dtype, int64_t ldo, int act,
                                 edg_stream stream) {
  return gate_rows_entry(h, dtype, ldh, sent_ptr, B, D, gate, out, out_dtype, ldo, act, stream);
}

extern "C" int edg_sigmoid_bwd(const void* y, int y_dtype, int64_t ldy, const void* dy, int dy_dtype,
                               int64_t lddy, int32_t R, int32_t C, void* dz, int dz_dtype, int64_t lddz,
                               int accumulate, edg_stream stream) {
  if (R < 0 || C <= 0) return EDG_ERR_ARG;
  if (R == 0) return EDG_OK;
  if (!y || !dy || !dz) return EDG_ERR_ARG;
  if (lddz < C) return EDG_ERR_ARG;
  sigmoid_bwd_kernel<<<blocks_for((int64_t)R * lddz, 256), 256, 0, (cudaStream_t)stream>>>(y, y_dtype, ldy, dy, dy_dtype, lddy, R, C, dz, dz_dtype, lddz, accumulate);
  return check_launch();
}

extern "C" int edg_cast_2d(const float* src, int64_t lds, int32_t R, int32_t C, void* dst, int dst_dtype,
                           int64_t ldd, int transpose, edg_stream stream) {
  if (R <= 0 || C <= 0 || !src || !dst) return EDG_ERR_ARG;
  const int rows_out = transpose ? C : R, cols_out = transpose ? R : C;
  if (ldd < cols_out) return EDG_ERR_ARG;
  if (dst_dtype != EDG_F32 && dst_dtype != EDG_BF16) return EDG_ERR_DTYPE;
  cast_2d_kernel<<<blocks_for((int64_t)rows_out * ldd, 256), 256, 0, (cudaStream_t)stream>>>(src, lds, R, C, dst, dst_dtype, ldd, transpose);
  return check_launch();
}

extern "C" int edg_cast_batch(int32_t n, const void* const* src, void* const* dst, const int32_t* R, const int32_t* C,
                              const int64_t* lds, const int64_t* ldd, const int32_t* transpose, int dst_dtype,
                              edg_stream stream) {
  if (n < 0 || n > kCastBatchMax) return EDG_ERR_UNSUPPORTED;
  if (n == 0) return EDG_OK;
  if (!src || !dst || !R || !C || !lds || !ldd || !transpose) return EDG_ERR_ARG;
  if (dst_dtype != EDG_F32 && dst_dtype != EDG_BF16) return EDG_ERR_DTYPE;
  CastBatch b;
  int64_t most = 0;
  for (int i = 0; i < n; ++i) {
    if (!src[i] || !dst[i] || R[i] <= 0 || C[i] <= 0) return EDG_ERR_ARG;
    const int cols_out = transpose[i] ? R[i] : C[i], rows_out = transpose[i] ? C[i] : R[i];
    if (ldd[i] < cols_out || ldd[i] > 0x7fffffff || lds[i] > 0x7fffffff) return EDG_ERR_ARG;
    b.src[i] = (const float*)src[i]; b.dst[i] = dst[i];
    b.R[i] = R[i]; b.C[i] = C[i]; b.lds[i] = (int)lds[i]; b.ldd[i] = (int)ldd[i]; b.transpose[i] = transpose[i];
    const int64_t tot = (int64_t)rows_out * ldd[i];
    if (tot > most) most = tot;
  }
  int bx = (int)((most + 255) / 256);
  if (bx > 128) bx = 128;
  cast_batch_kernel<<<dim3(bx, n), 256, 0, (cudaStream_t)stream>>>(b, dst_dtype);
  return check_launch();
}
