// FFMA GEMMs of the fp32-parity mode (SURVEY hard part 1: single-pass TF32 misses the
// 1e-5 bar, so the fp32 mode stays on the fp32 pipe).
//   linear: C[M,Nout] = act(A[M,K] * W[Nout,K]^T + bias)
//   wgrad : P[s][K1,K2] = sum_{r in split s} A[r,K1]^T B[r,K2]  (+ deterministic split reduce)
#include <type_traits>

#include "edg_common.cuh"

namespace edg {

constexpr int TM = 64, TN = 64, TK = 16;

template <typename T>
__device__ __forceinline__ void load4(const T* p, int64_t valid, float (&f)[4]) {
  // up to 4 consecutive elements, zero-filled past `valid`
#pragma unroll
  for (int i = 0; i < 4; ++i) f[i] = (i < valid) ? to_f32(p[i]) : 0.f;
}
template <>
__device__ __forceinline__ void load4<float>(const float* p, int64_t valid, float (&f)[4]) {
  if (valid >= 4 && ((reinterpret_cast<uintptr_t>(p) & 15u) == 0)) {
    float4 v = __ldg(reinterpret_cast<const float4*>(p));
    f[0] = v.x; f[1] = v.y; f[2] = v.z; f[3] = v.w;
  } else {
#pragma unroll
    for (int i = 0; i < 4; ++i) f[i] = (i < valid) ? p[i] : 0.f;
  }
}

template <typename TA, typename TC>
__global__ void __launch_bounds__(256)
linear_simt_kernel(const TA* __restrict__ A, int64_t lda, int M, int K, const TA* __restrict__ W, int64_t ldw,
                   int Nout, const float* __restrict__ bias, int act, TC* __restrict__ C, int64_t ldc) {
  __shared__ float As[TK][TM + 4];
  __shared__ float Ws[TK][TN + 4];
  const int tid = threadIdx.x;
  const int m0 = blockIdx.y * TM, n0 = blockIdx.x * TN;
  const int lr = tid >> 2, lk = (tid & 3) * 4;      // loader: row 0..63, k offset 0,4,8,12
  const int ty = tid >> 4, tx = tid & 15;           // compute: 4x4 micro tile
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

  for (int k0 = 0; k0 < K; k0 += TK) {
    float a[4], w[4];
    const int kk = k0 + lk;
    const int am = m0 + lr, wn = n0 + lr;
    if (am < M) load4<TA>(A + (int64_t)am * lda + kk, (int64_t)K - kk, a);
    else a[0] = a[1] = a[2] = a[3] = 0.f;
    if (wn < Nout) load4<TA>(W + (int64_t)wn * ldw + kk, (int64_t)K - kk, w);
    else w[0] = w[1] = w[2] = w[3] = 0.f;
#pragma unroll
    for (int i = 0; i < 4; ++i) { As[lk + i][lr] = a[i]; Ws[lk + i][lr] = w[i]; }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < TK; ++k) {
      const float4 av = *reinterpret_cast<const float4*>(&As[k][ty * 4]);
      const float4 wv = *reinterpret_cast<const float4*>(&Ws[k][tx * 4]);
      const float ar[4] = {av.x, av.y, av.z, av.w}, wr[4] = {wv.x, wv.y, wv.z, wv.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(ar[i], wr[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int m = m0 + ty * 4 + i;
    if (m >= M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int n = n0 + tx * 4 + j;
      if (n >= Nout) {
        if (n < ldc) C[(int64_t)m * ldc + n] = from_f32<TC>(0.f);   // keep row padding zero
        continue;
      }
      float v = acc[i][j] + (bias ? __ldg(bias + n) : 0.f);
      if (act == EDG_ACT_SIGMOID) v = sigmoidf_(v);
      else if (act == EDG_ACT_RELU) v = fmaxf(v, 0.f);
      C[(int64_t)m * ldc + n] = from_f32<TC>(v);
    }
  }
}

// partial[z][K1,K2] over rows [z*rows_per, ...)
template <typename T>
__global__ void __launch_bounds__(256)
wgrad_simt_kernel(const T* __restrict__ A, int64_t lda, int K1, const T* __restrict__ B, int64_t ldb, int K2,
                  int R, int rows_per, float* __restrict__ partial) {
  __shared__ float As[TK][TM + 4];
  __shared__ float Bs[TK][TN + 4];
  const int tid = threadIdx.x;
  const int m0 = blockIdx.y * TM, n0 = blockIdx.x * TN;
  const int r_beg = blockIdx.z * rows_per, r_end = min(R, r_beg + rows_per);
  const int lr = tid >> 4, lc = (tid & 15) * 4;     // loader: r 0..15, col offset 0..60
  const int ty = tid >> 4, tx = tid & 15;
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  for (int r0 = r_beg; r0 < r_end; r0 += TK) {
    const int r = r0 + lr;
    float a[4], b[4];
    if (r < r_end) {
      load4<T>(A + (int64_t)r * lda + m0 + lc, (int64_t)K1 - (m0 + lc), a);
      load4<T>(B + (int64_t)r * ldb + n0 + lc, (int64_t)K2 - (n0 + lc), b);
    } else {
      a[0] = a[1] = a[2] = a[3] = 0.f;
      b[0] = b[1] = b[2] = b[3] = 0.f;
    }
    *reinterpret_cast<float4*>(&As[lr][lc]) = make_float4(a[0], a[1], a[2], a[3]);
    *reinterpret_cast<float4*>(&Bs[lr][lc]) = make_float4(b[0], b[1], b[2], b[3]);
    __syncthreads();
#pragma unroll
    for (int k = 0; k < TK; ++k) {
      const float4 av = *reinterpret_cast<const float4*>(&As[k][ty * 4]);
      const float4 bv = *reinterpret_cast<const float4*>(&Bs[k][tx * 4]);
      const float ar[4] = {av.x, av.y, av.z, av.w}, br[4] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(ar[i], br[j], acc[i][j]);
    }
    __syncthreads();
  }
  float* P = partial + (int64_t)blockIdx.z * K1 * K2;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int m = m0 + ty * 4 + i;
    if (m >= K1) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int n = n0 + tx * 4 + j;
      if (n < K2) P[(int64_t)m * K2 + n] = acc[i][j];
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Large-tile fp32 variants (128 x 128 x 8, 8 x 8 register tiles, double-buffered shared memory, one barrier per
// K step): the 64 x 64 kernels above reach ~26 TFLOP/s at the dense-compat C2 shape ([204800, 300] x [300, 300]),
// which made the fp32 drop-in layer slower than torch's own cuBLAS formulation on the same GPU.  fp32 in, fp32
// accumulate, fp32 out -- the 1e-5 parity mode stays on the FFMA pipe (single-pass TF32 misses the bar).
// ---------------------------------------------------------------------------------------------------------------
constexpr int BM = 128, BN = 128, BK = 8, BP = BM + 4;      // BP: padded pitch of a shared-memory K row

// 64 FMAs per K step from four 128-bit shared loads
__device__ __forceinline__ void mma_8x8(const float (*As)[BP], const float (*Bs)[BP], int ty, int tx, float (&acc)[8][8]) {
#pragma unroll
  for (int k = 0; k < BK; ++k) {
    const float4 a0 = *reinterpret_cast<const float4*>(&As[k][ty * 4]);
    const float4 a1 = *reinterpret_cast<const float4*>(&As[k][64 + ty * 4]);
    const float4 b0 = *reinterpret_cast<const float4*>(&Bs[k][tx * 4]);
    const float4 b1 = *reinterpret_cast<const float4*>(&Bs[k][64 + tx * 4]);
    const float ar[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
    const float br[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(ar[i], br[j], acc[i][j]);
  }
}

__global__ void __launch_bounds__(256, 2)
linear_big_kernel(const float* __restrict__ A, int64_t lda, int M, int K, const float* __restrict__ W, int64_t ldw,
                  int Nout, const float* __restrict__ bias, int act, float* __restrict__ C, int64_t ldc, int zend) {
  // zend: columns [Nout, zend) are the row's own padding and are written as zeros; nothing is written past zend
  __shared__ __align__(16) float As[2][BK][BP];
  __shared__ __align__(16) float Ws[2][BK][BP];
  const int tid = threadIdx.x;
  const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;
  const int lr = tid >> 1, lk = (tid & 1) * 4;        // loader: tile row 0..127, k offset 0 / 4
  const int ty = tid >> 4, tx = tid & 15;
  const int am = m0 + lr, wn = n0 + lr;
  float acc[8][8];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
  float a[4], w[4];
  auto fetch = [&](int k0) {
    const int kk = k0 + lk;
    if (am < M && kk < K) load4<float>(A + (int64_t)am * lda + kk, (int64_t)K - kk, a);
    else a[0] = a[1] = a[2] = a[3] = 0.f;
    if (wn < Nout && kk < K) load4<float>(W + (int64_t)wn * ldw + kk, (int64_t)K - kk, w);
    else w[0] = w[1] = w[2] = w[3] = 0.f;
  };
  auto stash = [&](int buf) {
#pragma unroll
    for (int i = 0; i < 4; ++i) { As[buf][lk + i][lr] = a[i]; Ws[buf][lk + i][lr] = w[i]; }
  };
  fetch(0);
  stash(0);
  __syncthreads();
  int cur = 0;
  for (int k0 = 0; k0 < K; k0 += BK) {
    const bool more = k0 + BK < K;
    if (more) fetch(k0 + BK);                          // global loads of the next K step fly during the FMAs
    mma_8x8(As[cur], Ws[cur], ty, tx, acc);
    if (more) stash(cur ^ 1);
    __syncthreads();
    cur ^= 1;
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int m = m0 + (i < 4 ? ty * 4 + i : 64 + ty * 4 + i - 4);
    if (m >= M) continue;
    float* crow = C + (int64_t)m * ldc;
#pragma unroll
    for (int jg = 0; jg < 2; ++jg) {
      const int n = n0 + jg * 64 + tx * 4;
      float v[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int nj = n + j;
        float x = acc[i][jg * 4 + j] + ((bias && nj < Nout) ? __ldg(bias + nj) : 0.f);
        if (act == EDG_ACT_SIGMOID) x = sigmoidf_(x);
        else if (act == EDG_ACT_RELU) x = fmaxf(x, 0.f);
        v[j] = nj < Nout ? x : 0.f;                    // columns in [Nout, ldc) are row padding: kept zero
      }
      if (n + 4 <= zend && (ldc & 3) == 0) *reinterpret_cast<float4*>(crow + n) = make_float4(v[0], v[1], v[2], v[3]);
      else
#pragma unroll
        for (int j = 0; j < 4; ++j)
          if (n + j < zend) crow[n + j] = v[j];
    }
  }
}

__global__ void __launch_bounds__(256, 2)
wgrad_big_kernel(const float* __restrict__ A, int64_t lda, int K1, const float* __restrict__ B, int64_t ldb, int K2,
                 int R, int rows_per, float* __restrict__ partial) {
  __shared__ __align__(16) float As[2][BK][BP];
  __shared__ __align__(16) float Bs[2][BK][BP];
  const int tid = threadIdx.x;
  const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;
  const int r_beg = blockIdx.z * rows_per, r_end = min(R, r_beg + rows_per);
  const int lr = tid >> 5, lc = (tid & 31) * 4;        // loader: row 0..7 of the K step, 4 consecutive columns
  const int ty = tid >> 4, tx = tid & 15;
  float acc[8][8];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
  float a[4], b[4];
  auto fetch = [&](int r0) {
    const int r = r0 + lr;
    if (r < r_end && m0 + lc < K1) load4<float>(A + (int64_t)r * lda + m0 + lc, (int64_t)K1 - (m0 + lc), a);
    else a[0] = a[1] = a[2] = a[3] = 0.f;
    if (r < r_end && n0 + lc < K2) load4<float>(B + (int64_t)r * ldb + n0 + lc, (int64_t)K2 - (n0 + lc), b);
    else b[0] = b[1] = b[2] = b[3] = 0.f;
  };
  auto stash = [&](int buf) {
    *reinterpret_cast<float4*>(&As[buf][lr][lc]) = make_float4(a[0], a[1], a[2], a[3]);
    *reinterpret_cast<float4*>(&Bs[buf][lr][lc]) = make_float4(b[0], b[1], b[2], b[3]);
  };
  fetch(r_beg);
  stash(0);
  __syncthreads();
  int cur = 0;
  for (int r0 = r_beg; r0 < r_end; r0 += BK) {
    const bool more = r0 + BK < r_end;
    if (more) fetch(r0 + BK);
    mma_8x8(As[cur], Bs[cur], ty, tx, acc);
    if (more) stash(cur ^ 1);
    __syncthreads();
    cur ^= 1;
  }
  float* P = partial + (int64_t)blockIdx.z * K1 * K2;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int m = m0 + (i < 4 ? ty * 4 + i : 64 + ty * 4 + i - 4);
    if (m >= K1) continue;
#pragma unroll
    for (int jg = 0; jg < 2; ++jg) {
      const int n = n0 + jg * 64 + tx * 4;
      if (n + 4 <= K2 && (K2 & 3) == 0)
        *reinterpret_cast<float4*>(P + (int64_t)m * K2 + n) =
            make_float4(acc[i][jg * 4], acc[i][jg * 4 + 1], acc[i][jg * 4 + 2], acc[i][jg * 4 + 3]);
      else
#pragma unroll
        for (int j = 0; j < 4; ++j)
          if (n + j < K2) P[(int64_t)m * K2 + n + j] = acc[i][jg * 4 + j];
    }
  }
}

static bool big_linear_ok(int M, int K, int Nout) { return M >= 512 && Nout >= 96 && K >= 32; }
static bool big_wgrad_ok(int R, int K1, int K2) { return R >= 4096 && K1 >= 96 && K2 >= 96; }
static int wgrad_big_splits(int R, int K1, int K2) {
  const int tiles = ((K1 + BM - 1) / BM) * ((K2 + BN - 1) / BN);
  int want = (4 * kNumSMs + tiles - 1) / tiles;
  int maxs = (R + 511) / 512;          // at least 512 rows per split
  int s = want < maxs ? want : maxs;
  return s < 1 ? 1 : s;
}

// dW[m, n] (+)= sum_z partial[z][m*K2+n]   (fixed order -> deterministic)
__global__ void split_reduce_kernel(const float* __restrict__ partial, int splits, int K1, int K2,
                                    float* __restrict__ dW, int64_t lddw, int accumulate) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t tot = (int64_t)K1 * K2;
  if (idx >= tot) return;
  float s = 0.f;
  for (int z = 0; z < splits; ++z) s += partial[(int64_t)z * tot + idx];
  const int m = (int)(idx / K2), n = (int)(idx - (int64_t)m * K2);
  float* o = dW + (int64_t)m * lddw + n;
  *o = accumulate ? (*o + s) : s;
}

// ---- column sums ------------------------------------------------------------
constexpr int kColsumRowsPer = 1024;
template <typename T>
__global__ void colsum_partial_kernel(const T* __restrict__ x, int64_t ldx, int R, int C, float* __restrict__ partial) {
  // block = 32 columns x 8 row lanes; grid.y = row chunk
  __shared__ float red[8][33];
  const int c = blockIdx.x * 32 + (threadIdx.x & 31);
  const int ry = threadIdx.x >> 5;
  const int r_beg = blockIdx.y * kColsumRowsPer, r_end = min(R, r_beg + kColsumRowsPer);
  float s = 0.f;
  if (c < C)
    for (int r = r_beg + ry; r < r_end; r += 8) s += to_f32(x[(int64_t)r * ldx + c]);
  red[ry][threadIdx.x & 31] = s;
  __syncthreads();
  if (ry == 0 && c < C) {
    float t = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) t += red[i][threadIdx.x];
    partial[(int64_t)blockIdx.y * C + c] = t;
  }
}
__global__ void colsum_final_kernel(const float* __restrict__ partial, int chunks, int C, float* __restrict__ out, int accumulate) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  float s = 0.f;
  for (int k = 0; k < chunks; ++k) s += partial[(int64_t)k * C + c];
  out[c] = accumulate ? out[c] + s : s;
}

// one element summed over `slabs` partial-sum slabs `tot` floats apart: eight loads in flight, four chains (the plain
// loop has one load in flight per thread and is latency-bound: 54 -> 40 us at 444 slabs of 361 KB)
__device__ __forceinline__ float sum_slabs(const float* __restrict__ p, int slabs, int64_t tot) {
  float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
  int z = 0;
  for (; z + 8 <= slabs; z += 8) {
    float v[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) v[u] = __ldg(p + (int64_t)(z + u) * tot);
    s0 += v[0] + v[4]; s1 += v[1] + v[5]; s2 += v[2] + v[6]; s3 += v[3] + v[7];
  }
  for (; z < slabs; ++z) s0 += __ldg(p + (int64_t)z * tot);
  return (s0 + s1) + (s2 + s3);
}

// as split_reduce, for partials of extended shape [K1e, K2e] whose extra row (bias_of 2) or column (bias_of 1)
// holds the bias gradient
__global__ void split_reduce_bias_kernel(const float* __restrict__ partial, int splits, int K1, int K2, int K1e, int K2e,
                                         float* __restrict__ dW, int64_t lddw, float* __restrict__ dbias, int bias_of,
                                         int accumulate) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t tot = (int64_t)K1e * K2e;
  if (idx >= tot) return;
  const int m = (int)(idx / K2e), n = (int)(idx - (int64_t)m * K2e);
  const float s = sum_slabs(partial + idx, splits, tot);
  float* o = nullptr;
  if (m < K1 && n < K2) o = dW + (int64_t)m * lddw + n;
  else if (bias_of == 2 && m == K1 && n < K2) o = dbias + n;
  else if (bias_of == 1 && n == K2 && m < K1) o = dbias + m;
  if (o) *o = accumulate ? (*o + s) : s;
}

void launch_split_reduce_bias(const float* partial, int splits, int K1, int K2, int K1e, int K2e, float* dW, int64_t lddw,
                              float* dbias, int bias_of, int accumulate, cudaStream_t s) {
  const int64_t tot = (int64_t)K1e * K2e;
  split_reduce_bias_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, s>>>(partial, splits, K1, K2, K1e, K2e, dW, lddw, dbias,
                                                                         bias_of, accumulate);
}

// the same for n problems in one launch: blockIdx.y = problem, slabs [problem][split][K1e][K2e]
struct ReduceBatchPtrs { float* dW[8]; float* dbias[8]; };
__global__ void split_reduce_bias_batch_kernel(const float* __restrict__ partial, int splits, int K1, int K2, int K1e, int K2e,
                                               const __grid_constant__ ReduceBatchPtrs ptrs, int64_t lddw, int bias_of) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t tot = (int64_t)K1e * K2e;
  if (idx >= tot) return;
  const int p = blockIdx.y;
  const float* base = partial + (int64_t)p * splits * tot;
  const int m = (int)(idx / K2e), n = (int)(idx - (int64_t)m * K2e);
  const float s = sum_slabs(base + idx, splits, tot);
  if (m < K1 && n < K2) ptrs.dW[p][(int64_t)m * lddw + n] = s;
  else if (bias_of == 2 && m == K1 && n < K2) ptrs.dbias[p][n] = s;
  else if (bias_of == 1 && n == K2 && m < K1) ptrs.dbias[p][m] = s;
}

void launch_split_reduce_bias_batch(const float* partial, int n, int splits, int K1, int K2, int K1e, int K2e,
                                    float* const* dW, int64_t lddw, float* const* dbias, int bias_of, cudaStream_t s) {
  ReduceBatchPtrs ptrs;
  for (int i = 0; i < 8; ++i) { ptrs.dW[i] = i < n ? dW[i] : nullptr; ptrs.dbias[i] = (i < n && dbias) ? dbias[i] : nullptr; }
  const int64_t tot = (int64_t)K1e * K2e;
  split_reduce_bias_batch_kernel<<<dim3((unsigned)((tot + 255) / 256), n), 256, 0, s>>>(partial, splits, K1, K2, K1e, K2e, ptrs,
                                                                                        lddw, bias_of);
}

void launch_split_reduce(const float* partial, int splits, int K1, int K2, float* dW, int64_t lddw, int accumulate,
                         cudaStream_t s) {
  const int64_t tot = (int64_t)K1 * K2;
  split_reduce_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, s>>>(partial, splits, K1, K2, dW, lddw, accumulate);
}

int wgrad_splits(int R, int K1, int K2) {
  const int tiles = ((K1 + TM - 1) / TM) * ((K2 + TN - 1) / TN);
  int want = (4 * kNumSMs + tiles - 1) / tiles;
  int maxs = (R + 255) / 256;          // at least 256 rows per split
  int s = want < maxs ? want : maxs;
  return s < 1 ? 1 : s;
}

template <typename TA>
int launch_linear_simt(const void* A, int64_t lda, int M, int K, const void* W, int64_t ldw, int Nout,
                       const float* bias, int act, void* C, int c_dtype, int64_t ldc, cudaStream_t s) {
  const int ncols = (int)(ldc < (int64_t)Nout + 16 ? ldc : Nout);       // also covers the padding columns
  if (std::is_same<TA, float>::value && c_dtype == EDG_F32 && big_linear_ok(M, K, Nout)) {
    dim3 gb((ncols + BN - 1) / BN, (M + BM - 1) / BM);
    if (gb.y <= 65535) {
      linear_big_kernel<<<gb, 256, 0, s>>>((const float*)A, lda, M, K, (const float*)W, ldw, Nout, bias, act, (float*)C, ldc, ncols);
      return check_launch();
    }
  }
  dim3 grid((ncols + TN - 1) / TN, (M + TM - 1) / TM);
  if (grid.y > 65535) return EDG_ERR_UNSUPPORTED;
  if (c_dtype == EDG_F32)
    linear_simt_kernel<TA, float><<<grid, 256, 0, s>>>((const TA*)A, lda, M, K, (const TA*)W, ldw, Nout, bias, act, (float*)C, ldc);
  else
    linear_simt_kernel<TA, __nv_bfloat16><<<grid, 256, 0, s>>>((const TA*)A, lda, M, K, (const TA*)W, ldw, Nout, bias, act, (__nv_bfloat16*)C, ldc);
  return check_launch();
}
template int launch_linear_simt<float>(const void*, int64_t, int, int, const void*, int64_t, int, const float*, int, void*, int, int64_t, cudaStream_t);

template <typename T>
int launch_wgrad_simt(const void* A, int64_t lda, int K1, const void* B, int64_t ldb, int K2, int R,
                      float* dW, int64_t lddw, int accumulate, float* ws, cudaStream_t s) {
  if (std::is_same<T, float>::value && big_wgrad_ok(R, K1, K2)) {
    const int sb = wgrad_big_splits(R, K1, K2);
    int rp = (R + sb - 1) / sb;
    rp = ((rp + BK - 1) / BK) * BK;
    const int nsp = (R + rp - 1) / rp;
    dim3 gb((K2 + BN - 1) / BN, (K1 + BM - 1) / BM, nsp);
    wgrad_big_kernel<<<gb, 256, 0, s>>>((const float*)A, lda, K1, (const float*)B, ldb, K2, R, rp, ws);
    launch_split_reduce(ws, nsp, K1, K2, dW, lddw, accumulate, s);
    return check_launch();
  }
  const int splits = wgrad_splits(R, K1, K2);
  int rows_per = (R + splits - 1) / splits;
  rows_per = ((rows_per + TK - 1) / TK) * TK;
  dim3 grid((K2 + TN - 1) / TN, (K1 + TM - 1) / TM, splits);
  wgrad_simt_kernel<T><<<grid, 256, 0, s>>>((const T*)A, lda, K1, (const T*)B, ldb, K2, R, rows_per, ws);
  launch_split_reduce(ws, splits, K1, K2, dW, lddw, accumulate, s);
  return check_launch();
}
size_t wgrad_simt_workspace(int R, int K1, int K2) {
  int sp = wgrad_splits(R, K1, K2);
  if (big_wgrad_ok(R, K1, K2) && wgrad_big_splits(R, K1, K2) > sp) sp = wgrad_big_splits(R, K1, K2);
  return (size_t)sp * K1 * K2 * sizeof(float);
}
template int launch_wgrad_simt<float>(const void*, int64_t, int, const void*, int64_t, int, int, float*, int64_t, int, float*, cudaStream_t);

}  // namespace edg

using namespace edg;

extern "C" size_t edg_colsum_workspace(int32_t R, int32_t C) {
  if (R <= 0 || C <= 0) return 0;
  return (size_t)((R + kColsumRowsPer - 1) / kColsumRowsPer) * C * sizeof(float);
}

extern "C" int edg_colsum(const void* x, int dtype, int64_t ldx, int32_t R, int32_t C, float* out,
                          int accumulate, void* ws, size_t ws_bytes, edg_stream stream) {
  if (R < 0 || C <= 0 || !out) return EDG_ERR_ARG;
  cudaStream_t s = (cudaStream_t)stream;
  if (R == 0) {
    if (!accumulate) cudaMemsetAsync(out, 0, C * sizeof(float), s);
    return check_launch();
  }
  if (!x || !ws) return EDG_ERR_ARG;
  if (ws_bytes < edg_colsum_workspace(R, C)) return EDG_ERR_WORKSPACE;
  const int chunks = (R + kColsumRowsPer - 1) / kColsumRowsPer;
  dim3 grid((C + 31) / 32, chunks);
  if (chunks > 65535) return EDG_ERR_UNSUPPORTED;
  if (dtype == EDG_BF16)
    colsum_partial_kernel<__nv_bfloat16><<<grid, 256, 0, s>>>((const __nv_bfloat16*)x, ldx, R, C, (float*)ws);
  else if (dtype == EDG_F32)
    colsum_partial_kernel<float><<<grid, 256, 0, s>>>((const float*)x, ldx, R, C, (float*)ws);
  else return EDG_ERR_DTYPE;
  colsum_final_kernel<<<(C + 127) / 128, 128, 0, s>>>((const float*)ws, chunks, C, out, accumulate);
  return check_launch();
}
