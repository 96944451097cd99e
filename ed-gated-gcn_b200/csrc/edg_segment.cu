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
