// Segment reductions on the packed layout either side of the gated block (SURVEY 8f):
//   N1  word-piece -> word averaging: the dense `torch.bmm(transform, x)` of models/bert_amir5.py:600
//       (transform built at data_utils.py:438-451 with 1/l entries over contiguous word-piece runs)
//       as a segment MEAN over contiguous rows;
//   N4  BertDM's left / right dynamic max-pooling around the trigger (models/bertdm.py:116-140, :174-185).
// Both stream whole rows with 128-bit loads: HBM-bound, one pass.
#include <math.h>

#include <type_traits>

#include "edg_common.cuh"

namespace edg {

// ---- N1: y[i] = sum_{j in [start_i, start_i + len_i)} fl(1/len_i) * x[j] --------------------------------
template <typename TX, typename TY>
__global__ void __launch_bounds__(256)
segment_mean_kernel(const TX* __restrict__ x, int64_t ldx, const int32_t* __restrict__ seg_start,
                    const int32_t* __restrict__ seg_len, int N, int chunks, TY* __restrict__ y, int64_t ldy) {
  constexpr int E = Vec16<TX>::kElems;
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int i = (int)(idx / chunks);
  if (i >= N) return;
  const int c = (int)(idx - (int64_t)i * chunks) * E;
  const int beg = seg_start[i], len = seg_len[i];
  const float w = len > 0 ? __fdiv_rn(1.0f, (float)len) : 0.f;     // the fp32 transform entry (data_utils.py:449)
  float acc[E];
#pragma unroll
  for (int k = 0; k < E; ++k) acc[k] = 0.f;
  for (int j = 0; j < len; ++j) {                                   // ascending piece order, like the bmm row
    float f[E];
    Vec16<TX>::load(x + (int64_t)(beg + j) * ldx + c, f);
#pragma unroll
    for (int k = 0; k < E; ++k) acc[k] = fmaf(w, f[k], acc[k]);
  }
  TY* o = y + (int64_t)i * ldy + c;
  if constexpr (std::is_same<TX, TY>::value) {
    Vec16<TY>::store(o, acc);
  } else {
#pragma unroll
    for (int k = 0; k < E; ++k) o[k] = from_f32<TY>(acc[k]);
  }
}

// backward: dx[start_i + j] = fl(1/len_i) * dy[i]   (rows outside every segment are zeroed by the caller)
template <typename T>
__global__ void __launch_bounds__(256)
segment_mean_bwd_kernel(const T* __restrict__ dy, int64_t lddy, const int32_t* __restrict__ seg_start,
                        const int32_t* __restrict__ seg_len, int N, int chunks, T* __restrict__ dx, int64_t lddx) {
  constexpr int E = Vec16<T>::kElems;
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int i = (int)(idx / chunks);
  if (i >= N) return;
  const int c = (int)(idx - (int64_t)i * chunks) * E;
  const int beg = seg_start[i], len = seg_len[i];
  if (len <= 0) return;
  const float w = __fdiv_rn(1.0f, (float)len);
  float f[E];
  Vec16<T>::load(dy + (int64_t)i * lddy + c, f);
#pragma unroll
  for (int k = 0; k < E; ++k) f[k] *= w;
  for (int j = 0; j < len; ++j) Vec16<T>::store(dx + (int64_t)(beg + j) * lddx + c, f);
}

// ---- N4: left / right max-pool around the trigger -----------------------------------------------------
// bertdm.py:174-185:  L = x*maskL + 1, R = x*maskR + 1 over ALL T padded positions, max over t, then - 1.
// maskL = [t <= anchor], maskR = [anchor < t < n]; masked-out positions contribute 0 (+1): the left pool sees a
// zero when anchor + 1 < T, the right pool always does (position `anchor` itself).  torch.max returns the first
// index of the maximum: on the left the real rows come first (a real 0 beats the masked 0), on the right the
// masked zeros come first (a real row must be strictly positive to win).  arg = -1 when a masked zero wins
// (its gradient is multiplied by the mask, i.e. dropped).
template <typename T>
__global__ void __launch_bounds__(128)
lr_pool_fwd_kernel(const T* __restrict__ h, int64_t ldh, const int32_t* __restrict__ sent_ptr,
                   const int32_t* __restrict__ anchor, int B, int D, int chunks, int T_pad,
                   float* __restrict__ pooled, int32_t* __restrict__ arg) {
  constexpr int E = Vec16<T>::kElems;
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int b = (int)(idx / chunks);
  if (b >= B) return;
  const int c = (int)(idx - (int64_t)b * chunks) * E;
  const int beg = sent_ptr[b], end = sent_ptr[b + 1];
  const int a = anchor[b];
  const int split = min(end, beg + a + 1);           // rows [beg, split) are left of / at the trigger
  float mL[E], mR[E];
  int32_t wL[E], wR[E];
#pragma unroll
  for (int k = 0; k < E; ++k) { mL[k] = -INFINITY; mR[k] = 0.f; wL[k] = -1; wR[k] = -1; }
  for (int t = beg; t < split; ++t) {
    float f[E];
    Vec16<T>::load(h + (int64_t)t * ldh + c, f);
#pragma unroll
    for (int k = 0; k < E; ++k)
      if (f[k] > mL[k]) { mL[k] = f[k]; wL[k] = t; }
  }
  for (int t = split; t < end; ++t) {
    float f[E];
    Vec16<T>::load(h + (int64_t)t * ldh + c, f);
#pragma unroll
    for (int k = 0; k < E; ++k)
      if (f[k] > mR[k]) { mR[k] = f[k]; wR[k] = t; }
  }
  const bool zero_left = (a + 1 < T_pad) || (split == beg);
#pragma unroll
  for (int k = 0; k < E; ++k) {
    if (c + k >= D) break;
    if (zero_left && !(mL[k] >= 0.f)) { mL[k] = 0.f; wL[k] = -1; }
    const int64_t o = (int64_t)b * 2 * D + c + k;
    pooled[o] = __fsub_rn(__fadd_rn(mL[k], 1.0f), 1.0f);            // the reference's +1 / -1 (bertdm.py:176-183)
    pooled[o + D] = __fsub_rn(__fadd_rn(mR[k], 1.0f), 1.0f);
    arg[o] = wL[k];
    arg[o + D] = wR[k];
  }
}

// dh[arg[b,j], j mod D] += g[b,j]; a thread owns column (b, d) of both halves (distinct rows), so no two
// threads touch the same element.
template <typename T>
__global__ void __launch_bounds__(256)
lr_pool_bwd_kernel(const float* __restrict__ g, const int32_t* __restrict__ arg, int B, int D, T* __restrict__ dh,
                   int64_t lddh) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int b = (int)(idx / D);
  if (b >= B) return;
  const int d = (int)(idx - (int64_t)b * D);
#pragma unroll
  for (int s = 0; s < 2; ++s) {
    const int64_t o = (int64_t)b * 2 * D + s * D + d;
    const int32_t r = arg[o];
    if (r >= 0) {
      T* p = dh + (int64_t)r * lddh + d;
      *p = from_f32<T>(to_f32(*p) + g[o]);
    }
  }
}

// ---- N4 on grouped trigger pairs ------------------------------------------------------------------------------
// The rows of a sentence exist once; pair p of sentence s (pairs pair_ptr[s] .. pair_ptr[s+1] - 1, sentence-local
// anchor a_p) gets what lr_pool_fwd_kernel gives that pair's copy of the sentence, with arg naming the sentence row.
// The left pool of a pair is a prefix maximum of the sentence and the right pool a suffix maximum, so one block per
// (sentence, slab of 32 16-byte column chunks), a thread per chunk, reads the slab twice whatever the pair count:
//   ascending pass  (strict >: the first row of the maximum wins) -- emits the left half of every pair whose anchor
//                   it has just passed, against the masked zero as in lr_pool_fwd_kernel;
//   descending pass (>=: the smallest row wins ties, as the first index does in an ascending scan) -- emits the right
//                   half of every pair whose anchor it is about to pass; a real row wins only if strictly positive
//                   (the masked zeros come first in the reference's order).
// The pairs are visited in anchor order through a counting sort in shared memory.  A sentence longer than
// kLRPairsMaxLen rows or with more than kLRPairsMaxPairs pairs runs the per-pair scan of lr_pool_fwd_kernel instead,
// pair after pair in the same block.
constexpr int kLRPairsChunks = 32;       // threads (16-byte column chunks) per block: one warp
constexpr int kLRPairsMaxLen = 512;
constexpr int kLRPairsMaxPairs = 2048;
constexpr int kLRPairsBwdRows = 64;      // sentence rows per shared-memory tile of the backward

// one half (E columns at c) of a pair's output; vec: D % 4 == 0 and 16-byte aligned outputs
template <int E>
__device__ __forceinline__ void lr_pairs_emit(float* __restrict__ pooled, int32_t* __restrict__ arg, int64_t o, int c,
                                              int D, int vec, const float (&m)[E], const int32_t (&w)[E]) {
  if (vec && c + E <= D) {
#pragma unroll
    for (int k = 0; k < E; k += 4) {
      *reinterpret_cast<float4*>(pooled + o + k) = make_float4(m[k], m[k + 1], m[k + 2], m[k + 3]);
      *reinterpret_cast<int4*>(arg + o + k) = make_int4(w[k], w[k + 1], w[k + 2], w[k + 3]);
    }
  } else {
#pragma unroll
    for (int k = 0; k < E; ++k)
      if (c + k < D) { pooled[o + k] = m[k]; arg[o + k] = w[k]; }
  }
}

// lr_pool_fwd_kernel's scan for one pair (the path of sentences outside the shared-memory plan)
template <typename T>
__device__ void lr_pool_pair_scan(const T* __restrict__ h, int64_t ldh, int beg, int end, int a, int T_pad, int c, int D,
                                  int vec, float* __restrict__ pooled, int32_t* __restrict__ arg, int64_t o) {
  constexpr int E = Vec16<T>::kElems;
  const int split = beg + min(max(a + 1, 0), end - beg);
  float mL[E], mR[E];
  int32_t wL[E], wR[E];
#pragma unroll
  for (int k = 0; k < E; ++k) { mL[k] = -INFINITY; mR[k] = 0.f; wL[k] = -1; wR[k] = -1; }
  for (int t = beg; t < split; ++t) {
    float f[E];
    Vec16<T>::load(h + (int64_t)t * ldh + c, f);
#pragma unroll
    for (int k = 0; k < E; ++k)
      if (f[k] > mL[k]) { mL[k] = f[k]; wL[k] = t; }
  }
  for (int t = split; t < end; ++t) {
    float f[E];
    Vec16<T>::load(h + (int64_t)t * ldh + c, f);
#pragma unroll
    for (int k = 0; k < E; ++k)
      if (f[k] > mR[k]) { mR[k] = f[k]; wR[k] = t; }
  }
  const bool zero_left = (a + 1 < T_pad) || (split == beg);
#pragma unroll
  for (int k = 0; k < E; ++k) {
    if (zero_left && !(mL[k] >= 0.f)) { mL[k] = 0.f; wL[k] = -1; }
    mL[k] = __fsub_rn(__fadd_rn(mL[k], 1.0f), 1.0f);
    mR[k] = __fsub_rn(__fadd_rn(mR[k], 1.0f), 1.0f);
  }
  lr_pairs_emit<E>(pooled, arg, o, c, D, vec, mL, wL);
  lr_pairs_emit<E>(pooled, arg, o + D, c, D, vec, mR, wR);
}

template <typename T>
__global__ void __launch_bounds__(kLRPairsChunks)
lr_pool_pairs_fwd_kernel(const T* __restrict__ h, int64_t ldh, const int32_t* __restrict__ sent_ptr,
                         const int32_t* __restrict__ pair_ptr, const int32_t* __restrict__ anchor, int D, int chunks,
                         int T_pad, int vec, float* __restrict__ pooled, int32_t* __restrict__ arg) {
  constexpr int E = Vec16<T>::kElems;
  constexpr int U = 32 / E;                      // rows in flight per thread
  __shared__ int bucket[kLRPairsMaxLen + 1];     // after the sort: sorted pairs of anchor k = [bucket[k-1], bucket[k])
  __shared__ int order[kLRPairsMaxPairs];        // pair offsets (from p0) in anchor order
  const int s = blockIdx.x, lane = threadIdx.x;
  const int beg = __ldg(sent_ptr + s), n = __ldg(sent_ptr + s + 1) - beg;
  const int p0 = __ldg(pair_ptr + s), np = __ldg(pair_ptr + s + 1) - p0;
  if (np <= 0) return;
  const int ci = blockIdx.y * kLRPairsChunks + lane;
  const bool live = ci < chunks;
  const int c = ci * E;
  const int64_t D2 = 2 * (int64_t)D;
  if (n <= 0 || n > kLRPairsMaxLen || np > kLRPairsMaxPairs) {
    if (!live) return;
    for (int p = p0; p < p0 + np; ++p)
      lr_pool_pair_scan<T>(h, ldh, beg, beg + n, __ldg(anchor + p), T_pad, c, D, vec, pooled, arg, p * D2 + c);
    return;
  }
  // counting sort by anchor (clamped into the sentence: an anchor past the end pools the whole sentence on the left)
  for (int i = lane; i <= n; i += kLRPairsChunks) bucket[i] = 0;
  __syncthreads();
  for (int i = lane; i < np; i += kLRPairsChunks) atomicAdd(&bucket[min(max(__ldg(anchor + p0 + i), 0), n - 1) + 1], 1);
  __syncthreads();
  {                                              // inclusive scan of bucket[0..n] by the warp: bucket[k] = first slot of k
    const int m = (n + kLRPairsChunks) / kLRPairsChunks, lo = lane * m, hi = min(lo + m, n + 1);
    int run = 0;
    for (int i = lo; i < hi; ++i) { run += bucket[i]; bucket[i] = run; }
    int off = run;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const int v = __shfl_up_sync(0xffffffffu, off, d);
      if (lane >= d) off += v;
    }
    off -= run;
    for (int i = lo; i < hi; ++i) bucket[i] += off;
  }
  __syncthreads();
  for (int i = lane; i < np; i += kLRPairsChunks)    // bucket[k] moves from the first slot of k to the first of k + 1
    order[atomicAdd(&bucket[min(max(__ldg(anchor + p0 + i), 0), n - 1)], 1)] = i;
  __syncthreads();
  if (!live) return;

  const T* hs = h + (int64_t)beg * ldh + c;
  float m[E];
  int32_t w[E];
#pragma unroll
  for (int k = 0; k < E; ++k) { m[k] = -INFINITY; w[k] = -1; }
  for (int t0 = 0; t0 < n; t0 += U) {            // ascending: left halves
    float f[U][E];
#pragma unroll
    for (int u = 0; u < U; ++u)
      if (t0 + u < n) Vec16<T>::load(hs + (int64_t)(t0 + u) * ldh, f[u]);
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int t = t0 + u;
      if (t >= n) break;
#pragma unroll
      for (int k = 0; k < E; ++k)
        if (f[u][k] > m[k]) { m[k] = f[u][k]; w[k] = beg + t; }
      for (int q = t ? bucket[t - 1] : 0; q < bucket[t]; ++q) {
        const int p = p0 + order[q];
        const bool zero_left = __ldg(anchor + p) + 1 < T_pad;
        float v[E];
        int32_t r[E];
#pragma unroll
        for (int k = 0; k < E; ++k) {
          const bool z = zero_left && !(m[k] >= 0.f);
          v[k] = __fsub_rn(__fadd_rn(z ? 0.f : m[k], 1.0f), 1.0f);
          r[k] = z ? -1 : w[k];
        }
        lr_pairs_emit<E>(pooled, arg, p * D2 + c, c, D, vec, v, r);
      }
    }
  }
#pragma unroll
  for (int k = 0; k < E; ++k) { m[k] = -INFINITY; w[k] = -1; }
  for (int t1 = n; t1 > 0; t1 -= U) {            // descending: right halves, emitted before their anchor row joins
    float f[U][E];
#pragma unroll
    for (int u = 0; u < U; ++u)
      if (t1 - 1 - u >= 0) Vec16<T>::load(hs + (int64_t)(t1 - 1 - u) * ldh, f[u]);
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int t = t1 - 1 - u;
      if (t < 0) break;
      const int q1 = bucket[t];
      int q = t ? bucket[t - 1] : 0;
      if (q < q1) {
        float v[E];
        int32_t r[E];
#pragma unroll
        for (int k = 0; k < E; ++k) {
          const bool real = m[k] > 0.f;
          v[k] = __fsub_rn(__fadd_rn(real ? m[k] : 0.f, 1.0f), 1.0f);
          r[k] = real ? w[k] : -1;
        }
        for (; q < q1; ++q) lr_pairs_emit<E>(pooled, arg, (p0 + order[q]) * D2 + D + c, c, D, vec, v, r);
      }
#pragma unroll
      for (int k = 0; k < E; ++k)
        if (f[u][k] >= m[k]) { m[k] = f[u][k]; w[k] = beg + t; }
    }
  }
}

// dh[t, c] = sum over the sentence's pairs p, ascending, of [argL_p,c = t] gL_p,c then [argR_p,c = t] gR_p,c, summed in
// one thread and rounded once: in fp64 for fp32 output (a row that holds the maximum for hundreds of pairs would otherwise
// carry hundreds of fp32 roundings), in fp32 for bf16 output.  One block per (sentence, slab of 32 chunks) as in the forward; the sentence is
// taken kLRPairsBwdRows rows at a time, each tile reading the pairs' g / arg once into a shared-memory accumulator
// column private to its thread ([row][k][lane]: no synchronisation, no bank conflicts).  Every row of every sentence
// is written (0 where nothing routes), padding columns up to the chunk end included.
template <typename T>
__global__ void __launch_bounds__(kLRPairsChunks)
lr_pool_pairs_bwd_kernel(const float* __restrict__ g, const int32_t* __restrict__ arg, const int32_t* __restrict__ sent_ptr,
                         const int32_t* __restrict__ pair_ptr, int D, int chunks, int vec, T* __restrict__ dh,
                         int64_t lddh) {
  constexpr int E = Vec16<T>::kElems;
  constexpr int U = 16 / E;                      // pairs in flight per thread
  using Acc = typename std::conditional<std::is_same<T, float>::value, double, float>::type;
  extern __shared__ __align__(16) unsigned char lr_acc[];
  const int lane = threadIdx.x, ci = blockIdx.y * kLRPairsChunks + lane;
  if (ci >= chunks) return;
  const int c = ci * E, s = blockIdx.x;
  const int beg = __ldg(sent_ptr + s), n = __ldg(sent_ptr + s + 1) - beg;
  const int p0 = __ldg(pair_ptr + s), p1 = __ldg(pair_ptr + s + 1);
  const int64_t D2 = 2 * (int64_t)D;
  Acc* acc = reinterpret_cast<Acc*>(lr_acc) + lane;   // element (r, k) at acc[(r * E + k) * 32]
  for (int t0 = 0; t0 < n; t0 += kLRPairsBwdRows) {
    const int rows = min(kLRPairsBwdRows, n - t0), lo = beg + t0;
    for (int i = 0; i < rows * E; ++i) acc[i * 32] = 0;
    for (int p = p0; p < p1; p += U) {
      float gv[U][2][E];
      int32_t av[U][2][E];
#pragma unroll
      for (int u = 0; u < U; ++u)
#pragma unroll
        for (int half = 0; half < 2; ++half) {
          const int64_t o = (p + u) * D2 + half * D + c;
          if (p + u < p1 && vec && c + E <= D) {
#pragma unroll
            for (int k = 0; k < E; k += 4) {
              const float4 x = __ldg(reinterpret_cast<const float4*>(g + o + k));
              const int4 y = __ldg(reinterpret_cast<const int4*>(arg + o + k));
              gv[u][half][k] = x.x; gv[u][half][k + 1] = x.y; gv[u][half][k + 2] = x.z; gv[u][half][k + 3] = x.w;
              av[u][half][k] = y.x; av[u][half][k + 1] = y.y; av[u][half][k + 2] = y.z; av[u][half][k + 3] = y.w;
            }
          } else {
#pragma unroll
            for (int k = 0; k < E; ++k) {
              const bool ok = p + u < p1 && c + k < D;
              gv[u][half][k] = ok ? __ldg(g + o + k) : 0.f;
              av[u][half][k] = ok ? __ldg(arg + o + k) : -1;
            }
          }
        }
#pragma unroll
      for (int u = 0; u < U; ++u)
#pragma unroll
        for (int half = 0; half < 2; ++half)
#pragma unroll
          for (int k = 0; k < E; ++k) {
            const int r = av[u][half][k] - lo;
            if ((unsigned)r < (unsigned)rows) acc[(r * E + k) * 32] += (Acc)gv[u][half][k];
          }
    }
    for (int r = 0; r < rows; ++r) {
      float f[E];
#pragma unroll
      for (int k = 0; k < E; ++k) f[k] = (float)acc[(r * E + k) * 32];
      Vec16<T>::store(dh + (int64_t)(lo + r) * lddh + c, f);
    }
  }
}

}  // namespace edg

using namespace edg;

extern "C" int edg_segment_mean(const void* x, int dtype, int64_t ldx, const int32_t* seg_start, const int32_t* seg_len,
                                int32_t N, int32_t D, void* y, int y_dtype, int64_t ldy, edg_stream stream) {
  if (N < 0 || D <= 0) return EDG_ERR_ARG;
  if (N == 0) return EDG_OK;
  if (!x || !seg_start || !seg_len || !y || ldx < D || ldy < D) return EDG_ERR_ARG;
  if (!aligned16(x) || !row_pitch_ok(dtype, ldx) || !aligned16(y) || !row_pitch_ok(y_dtype, ldy)) return EDG_ERR_ALIGN;
  cudaStream_t s = (cudaStream_t)stream;
  const int E = dtype == EDG_BF16 ? 8 : 4;
  const int chunks = (D + E - 1) / E;
  if ((int64_t)chunks * E > ldy || (int64_t)chunks * E > ldx) return EDG_ERR_ALIGN;
  const int64_t total = (int64_t)N * chunks;
  const unsigned grid = (unsigned)((total + 255) / 256);
  if (dtype == EDG_F32 && y_dtype == EDG_F32)
    segment_mean_kernel<float, float><<<grid, 256, 0, s>>>((const float*)x, ldx, seg_start, seg_len, N, chunks, (float*)y, ldy);
  else if (dtype == EDG_BF16 && y_dtype == EDG_BF16)
    segment_mean_kernel<__nv_bfloat16, __nv_bfloat16><<<grid, 256, 0, s>>>((const __nv_bfloat16*)x, ldx, seg_start, seg_len, N,
                                                                          chunks, (__nv_bfloat16*)y, ldy);
  else if (dtype == EDG_F32 && y_dtype == EDG_BF16)
    segment_mean_kernel<float, __nv_bfloat16><<<grid, 256, 0, s>>>((const float*)x, ldx, seg_start, seg_len, N, chunks,
                                                                  (__nv_bfloat16*)y, ldy);
  else if (dtype == EDG_BF16 && y_dtype == EDG_F32)
    segment_mean_kernel<__nv_bfloat16, float><<<grid, 256, 0, s>>>((const __nv_bfloat16*)x, ldx, seg_start, seg_len, N, chunks,
                                                                  (float*)y, ldy);
  else
    return EDG_ERR_DTYPE;
  return check_launch();
}

extern "C" int edg_segment_mean_bwd(const void* dy, int dtype, int64_t lddy, const int32_t* seg_start,
                                    const int32_t* seg_len, int32_t N, int32_t D, void* dx, int64_t lddx, int32_t P,
                                    edg_stream stream) {
  if (N < 0 || D <= 0 || P < 0) return EDG_ERR_ARG;
  if (P == 0) return EDG_OK;
  if (!dx || lddx < D) return EDG_ERR_ARG;
  if (!aligned16(dx) || !row_pitch_ok(dtype, lddx)) return EDG_ERR_ALIGN;
  if (dtype != EDG_F32 && dtype != EDG_BF16) return EDG_ERR_DTYPE;
  cudaStream_t s = (cudaStream_t)stream;
  // rows that belong to no word ([CLS], [SEP], padding pieces) receive no gradient
  if (cudaMemsetAsync(dx, 0, (size_t)P * lddx * dtype_size(dtype), s) != cudaSuccess) return check_launch();
  if (N == 0) return EDG_OK;
  if (!dy || !seg_start || !seg_len || lddy < D) return EDG_ERR_ARG;
  if (!aligned16(dy) || !row_pitch_ok(dtype, lddy)) return EDG_ERR_ALIGN;
  const int E = dtype == EDG_BF16 ? 8 : 4;
  const int chunks = (D + E - 1) / E;
  if ((int64_t)chunks * E > lddy || (int64_t)chunks * E > lddx) return EDG_ERR_ALIGN;
  const int64_t total = (int64_t)N * chunks;
  const unsigned grid = (unsigned)((total + 255) / 256);
  if (dtype == EDG_F32)
    segment_mean_bwd_kernel<float><<<grid, 256, 0, s>>>((const float*)dy, lddy, seg_start, seg_len, N, chunks, (float*)dx, lddx);
  else
    segment_mean_bwd_kernel<__nv_bfloat16><<<grid, 256, 0, s>>>((const __nv_bfloat16*)dy, lddy, seg_start, seg_len, N, chunks,
                                                               (__nv_bfloat16*)dx, lddx);
  return check_launch();
}

extern "C" int edg_lr_pool_fwd(const void* h, int dtype, int64_t ldh, const int32_t* sent_ptr, const int32_t* anchor,
                               int32_t B, int32_t D, int32_t T_pad, float* pooled, int32_t* arg, edg_stream stream) {
  if (B < 0 || D <= 0 || T_pad < 0) return EDG_ERR_ARG;
  if (B == 0) return EDG_OK;
  if (!h || !sent_ptr || !anchor || !pooled || !arg || ldh < D) return EDG_ERR_ARG;
  if (!aligned16(h) || !row_pitch_ok(dtype, ldh)) return EDG_ERR_ALIGN;
  cudaStream_t s = (cudaStream_t)stream;
  const int E = dtype == EDG_BF16 ? 8 : 4;
  const int chunks = (D + E - 1) / E;
  if ((int64_t)chunks * E > ldh) return EDG_ERR_ALIGN;
  const int64_t total = (int64_t)B * chunks;
  const unsigned grid = (unsigned)((total + 127) / 128);
  if (dtype == EDG_F32)
    lr_pool_fwd_kernel<float><<<grid, 128, 0, s>>>((const float*)h, ldh, sent_ptr, anchor, B, D, chunks, T_pad, pooled, arg);
  else if (dtype == EDG_BF16)
    lr_pool_fwd_kernel<__nv_bfloat16><<<grid, 128, 0, s>>>((const __nv_bfloat16*)h, ldh, sent_ptr, anchor, B, D, chunks, T_pad,
                                                          pooled, arg);
  else
    return EDG_ERR_DTYPE;
  return check_launch();
}

extern "C" int edg_lr_pool_bwd(const float* g, const int32_t* arg, int32_t B, int32_t D, void* dh, int dtype,
                               int64_t lddh, edg_stream stream) {
  if (B < 0 || D <= 0) return EDG_ERR_ARG;
  if (B == 0) return EDG_OK;
  if (!g || !arg || !dh || lddh < D) return EDG_ERR_ARG;
  cudaStream_t s = (cudaStream_t)stream;
  const int64_t total = (int64_t)B * D;
  const unsigned grid = (unsigned)((total + 255) / 256);
  if (dtype == EDG_F32) lr_pool_bwd_kernel<float><<<grid, 256, 0, s>>>(g, arg, B, D, (float*)dh, lddh);
  else if (dtype == EDG_BF16) lr_pool_bwd_kernel<__nv_bfloat16><<<grid, 256, 0, s>>>(g, arg, B, D, (__nv_bfloat16*)dh, lddh);
  else return EDG_ERR_DTYPE;
  return check_launch();
}

extern "C" int edg_lr_pool_pairs_fwd(const void* h, int dtype, int64_t ldh, const int32_t* sent_ptr, const int32_t* pair_ptr,
                                     const int32_t* anchor, int32_t S, int32_t P, int32_t D, int32_t T_pad, float* pooled,
                                     int32_t* arg, edg_stream stream) {
  if (S < 0 || P < 0 || D <= 0 || T_pad < 0) return EDG_ERR_ARG;
  if (S == 0 || P == 0) return EDG_OK;
  if (!h || !sent_ptr || !pair_ptr || !anchor || !pooled || !arg || ldh < D) return EDG_ERR_ARG;
  if (!aligned16(h) || !row_pitch_ok(dtype, ldh)) return EDG_ERR_ALIGN;
  cudaStream_t s = (cudaStream_t)stream;
  const int E = dtype == EDG_BF16 ? 8 : 4;
  const int chunks = (D + E - 1) / E;
  if ((int64_t)chunks * E > ldh) return EDG_ERR_ALIGN;
  const int vec = D % 4 == 0 && aligned16(pooled) && aligned16(arg);
  const dim3 grid((unsigned)S, (unsigned)((chunks + kLRPairsChunks - 1) / kLRPairsChunks));
  EDG_DISPATCH_T(dtype, lr_pool_pairs_fwd_kernel<T><<<grid, kLRPairsChunks, 0, s>>>(
      (const T*)h, ldh, sent_ptr, pair_ptr, anchor, D, chunks, T_pad, vec, pooled, arg);)
  return check_launch();
}

extern "C" int edg_lr_pool_pairs_bwd(const float* g, const int32_t* arg, const int32_t* sent_ptr, const int32_t* pair_ptr,
                                     int32_t S, int32_t P, int32_t D, void* dh, int dtype, int64_t lddh, edg_stream stream) {
  if (S < 0 || P < 0 || D <= 0) return EDG_ERR_ARG;
  if (S == 0) return EDG_OK;
  if (!sent_ptr || !pair_ptr || !dh || lddh < D || (P > 0 && (!g || !arg))) return EDG_ERR_ARG;
  if (!aligned16(dh) || !row_pitch_ok(dtype, lddh)) return EDG_ERR_ALIGN;
  cudaStream_t s = (cudaStream_t)stream;
  const int E = dtype == EDG_BF16 ? 8 : 4;
  const int chunks = (D + E - 1) / E;
  if ((int64_t)chunks * E > lddh) return EDG_ERR_ALIGN;
  const int vec = D % 4 == 0 && aligned16(g) && aligned16(arg);
  const dim3 grid((unsigned)S, (unsigned)((chunks + kLRPairsChunks - 1) / kLRPairsChunks));
  EDG_DISPATCH_T(dtype, {
    const size_t smem = (size_t)kLRPairsBwdRows * Vec16<T>::kElems * kLRPairsChunks * (std::is_same<T, float>::value ? 8 : 4);
    const int rc = ensure_dyn_smem((const void*)lr_pool_pairs_bwd_kernel<T>, smem);
    if (rc != EDG_OK) return rc;
    lr_pool_pairs_bwd_kernel<T><<<grid, kLRPairsChunks, smem, s>>>(g, arg, sent_ptr, pair_ptr, D, chunks, vec, (T*)dh, lddh);
  })
  return check_launch();
}

// ---------------------------------------------------------------------------------------------------------------
// Gate dropout (bert_amir5.py:624-625: `gate = self.dropout(gate)` on the gate BROADCAST to [B,T,D], i.e. an
// independent keep/drop decision per (token, column), shared by every use of that gate).  Since
// h * (gate * m * s) == (h * m * s) * gate, the per-token mask is applied to the ROWS once,
//     y[t,d] (+)= x[t,d] * keep(t,d) / (1 - p),
// and every kernel of the gated block then runs unchanged on the masked rows; the backward pass multiplies the row
// gradient by the same mask, regenerated from the seed (nothing is stored).
// keep(t,d) is a counter-based hash of (seed, stream, row, column) (edg_common.cuh, dropout_keep).
namespace edg {

template <typename T>
__global__ void __launch_bounds__(256)
dropout_rows_kernel(const T* __restrict__ x, int64_t ldx, T* __restrict__ y, int64_t ldy, int N, int D, int chunks,
                    const int64_t* __restrict__ seed, uint32_t stream_id, uint32_t thr, float scale, int accumulate) {
  constexpr int E = Vec16<T>::kElems;
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int row = (int)(idx / chunks);
  if (row >= N) return;
  const int c = (int)(idx - (int64_t)row * chunks) * E;
  const DropKey key = dropout_key(seed, stream_id);
  float f[E], o[E];
  Vec16<T>::load(x + (int64_t)row * ldx + c, f);
  if (accumulate) Vec16<T>::load(y + (int64_t)row * ldy + c, o);
#pragma unroll
  for (int k = 0; k < E; ++k) {
    const float v = (c + k < D && dropout_keep(key, (uint32_t)row, (uint32_t)(c + k), thr)) ? f[k] * scale : 0.f;
    o[k] = accumulate ? o[k] + v : v;
  }
  Vec16<T>::store(y + (int64_t)row * ldy + c, o);
}

}  // namespace edg

extern "C" int edg_dropout_rows(const void* x, int dtype, int64_t ldx, void* y, int64_t ldy, int32_t N, int32_t D,
                                const int64_t* seed, int32_t stream_id, float p, int accumulate, edg_stream stream) {
  if (N < 0 || D <= 0 || !edg::dropout_p_ok(p)) return EDG_ERR_ARG;
  if (N == 0) return EDG_OK;
  if (!x || !y || !seed || ldx < D || ldy < D) return EDG_ERR_ARG;
  if (!edg::aligned16(x) || !edg::aligned16(y) || !edg::row_pitch_ok(dtype, ldx) || !edg::row_pitch_ok(dtype, ldy)) return EDG_ERR_ALIGN;
  const int E = dtype == EDG_BF16 ? 8 : 4;
  const int chunks = (D + E - 1) / E;
  if ((int64_t)chunks * E > ldx || (int64_t)chunks * E > ldy) return EDG_ERR_ALIGN;
  const uint32_t thr = edg::dropout_threshold(p);
  const float scale = 1.0f / (1.0f - p);
  const int64_t total = (int64_t)N * chunks;
  const unsigned grid = (unsigned)((total + 255) / 256);
  cudaStream_t s = (cudaStream_t)stream;
  if (dtype == EDG_F32)
    edg::dropout_rows_kernel<float><<<grid, 256, 0, s>>>((const float*)x, ldx, (float*)y, ldy, N, D, chunks, seed, (uint32_t)stream_id,
                                                         thr, scale, accumulate);
  else if (dtype == EDG_BF16)
    edg::dropout_rows_kernel<__nv_bfloat16><<<grid, 256, 0, s>>>((const __nv_bfloat16*)x, ldx, (__nv_bfloat16*)y, ldy, N, D, chunks,
                                                                 seed, (uint32_t)stream_id, thr, scale, accumulate);
  else
    return EDG_ERR_DTYPE;
  return edg::check_launch();
}
