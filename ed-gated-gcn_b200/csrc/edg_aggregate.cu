// K2: degree-normalised neighbour aggregation over the packed CSR of many sentences
// (the `adj @ hidden / (rowsum + 1)` half of models/gcn.py:35,41).
//
// HBM-bound (about 1.5 flop/byte).  Work is flattened to (row, 16-byte chunk): consecutive
// threads read consecutive 128-bit chunks of one hidden row, then of the next row, so every
// request is a fully used 32-byte sector stream.  A row's neighbours live in the same
// sentence (a few KB away), so the 2-3 extra row reads per output row hit L1/L2; compulsory
// DRAM traffic is one read + one write of the [N,D] matrix plus 16 B/row of CSR.
#include "edg_staged.cuh"

namespace edg {

template <typename TO, int E>
__device__ __forceinline__ void store_chunk(TO* p, const float (&f)[E]);
template <> __device__ __forceinline__ void store_chunk<float, 4>(float* p, const float (&f)[4]) {
  *reinterpret_cast<float4*>(p) = make_float4(f[0], f[1], f[2], f[3]);
}
template <> __device__ __forceinline__ void store_chunk<float, 8>(float* p, const float (&f)[8]) {
  reinterpret_cast<float4*>(p)[0] = make_float4(f[0], f[1], f[2], f[3]);
  reinterpret_cast<float4*>(p)[1] = make_float4(f[4], f[5], f[6], f[7]);
}
template <> __device__ __forceinline__ void store_chunk<__nv_bfloat16, 8>(__nv_bfloat16* p, const float (&f)[8]) {
  Vec16<__nv_bfloat16>::store(p, f);
}
template <> __device__ __forceinline__ void store_chunk<__nv_bfloat16, 4>(__nv_bfloat16* p, const float (&f)[4]) {
  __nv_bfloat162 a = __floats2bfloat162_rn(f[0], f[1]), b = __floats2bfloat162_rn(f[2], f[3]);
  *reinterpret_cast<uint2*>(p) = make_uint2(*reinterpret_cast<uint32_t*>(&a), *reinterpret_cast<uint32_t*>(&b));
}

template <typename TI, typename TO, int MODE>
__global__ void __launch_bounds__(256)
aggregate_flat_kernel(const TI* __restrict__ x, int64_t ldx, TO* __restrict__ y, int64_t ldy, int N, int chunks,
                 const int32_t* __restrict__ row_ptr, const int32_t* __restrict__ col) {
  constexpr int E = Vec16<TI>::kElems;
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int row = (int)(idx / chunks);
  if (row >= N) return;
  const int c = (int)(idx - (int64_t)row * chunks) * E;
  const int beg = __ldg(row_ptr + row), end = __ldg(row_ptr + row + 1);
  float acc[E];
#pragma unroll
  for (int k = 0; k < E; ++k) acc[k] = 0.f;
  for (int e = beg; e < end; e += 4) {
    int nb[4];
    float w[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      nb[u] = (e + u < end) ? __ldg(col + e + u) : -1;
      w[u] = 1.f;
    }
    if (MODE == 1) {
#pragma unroll
      for (int u = 0; u < 4; ++u)
        if (nb[u] >= 0) w[u] = 1.0f / (float)(__ldg(row_ptr + nb[u] + 1) - __ldg(row_ptr + nb[u]) + 1);
    }
    float v[4][E];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      if (nb[u] >= 0) Vec16<TI>::load(x + (int64_t)nb[u] * ldx + c, v[u]);
      else {
#pragma unroll
        for (int k = 0; k < E; ++k) v[u][k] = 0.f;
      }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
#pragma unroll
      for (int k = 0; k < E; ++k) acc[k] = (MODE == 1) ? fmaf(v[u][k], w[u], acc[k]) : acc[k] + v[u][k];
    }
  }
  if (MODE == 0) {
    const float den = (float)(end - beg + 1);     // rowsum(adj) + 1, gcn.py:35
#pragma unroll
    for (int k = 0; k < E; ++k) acc[k] = acc[k] / den;
  }
  store_chunk<TO, E>(y + (int64_t)row * ldy + c, acc);
}

// ---- shared-memory staged variant ------------------------------------------------------------
// A block owns the sentences that START inside a window of `tile_rows` packed rows.  Those
// sentences' rows are contiguous in memory, so ONE bulk asynchronous copy (cp.async.bulk, TMA
// engine, mbarrier completion) stages them in shared memory; every neighbour of a staged row is
// in the same sentence, hence also staged: the gathers are 128-bit shared-memory loads and each
// hidden row leaves HBM/L2 exactly once.  Several blocks per SM overlap copy and gather.
__device__ __forceinline__ uint32_t agg_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// rows [r0, r1) straight from global memory (window overflow: a sentence longer than the buffer, or a
// non-tree graph with more than 4 non-zeros per row on average)
template <typename TI, typename TO, int MODE>
__device__ __noinline__ void aggregate_rows_global(const TI* __restrict__ x, int64_t ldx, TO* __restrict__ y, int64_t ldy,
                                                   int r0, int r1, const int32_t* __restrict__ row_ptr,
                                                   const int32_t* __restrict__ col) {
  constexpr int E = Vec16<TI>::kElems;
  const int c = threadIdx.x * E;
  for (int row = r0 + threadIdx.y; row < r1; row += blockDim.y) {
    const int beg = __ldg(row_ptr + row), end = __ldg(row_ptr + row + 1);
    float acc[E];
#pragma unroll
    for (int k = 0; k < E; ++k) acc[k] = 0.f;
    for (int e = beg; e < end; ++e) {
      const int j = __ldg(col + e);
      float v[E];
      Vec16<TI>::load(x + (int64_t)j * ldx + c, v);
      const float w = (MODE == 1) ? __frcp_rn((float)(__ldg(row_ptr + j + 1) - __ldg(row_ptr + j) + 1)) : 1.f;
#pragma unroll
      for (int k = 0; k < E; ++k) acc[k] = fmaf(v[k], w, acc[k]);
    }
    if (MODE == 0) {
      const float inv = __frcp_rn((float)(end - beg + 1));
#pragma unroll
      for (int k = 0; k < E; ++k) acc[k] *= inv;
    }
    store_chunk<TO, E>(y + (int64_t)row * ldy + c, acc);
  }
}

// MAXT is compile-time so that the default instantiation (384-thread blocks) does not carry the 64-register cap of
// 1024-thread blocks (it costs ~2-4 us per launch at C2)
template <typename TI, typename TO, int MODE, int MAXT>
__global__ void __launch_bounds__(MAXT)
aggregate_staged_kernel(const TI* __restrict__ x, int64_t ldx, TO* __restrict__ y, int64_t ldy, int N, int B,
                        int tile_rows, int cap_rows, const int32_t* __restrict__ sent_ptr,
                        const int32_t* __restrict__ row_sent, const int32_t* __restrict__ row_ptr,
                        const int32_t* __restrict__ col) {
  constexpr int E = Vec16<TI>::kElems;
  extern __shared__ __align__(128) uint8_t agg_smem[];
  __shared__ __align__(8) uint64_t bar;
  __shared__ int range[2];
  const int nthreads = blockDim.x * blockDim.y;
  const int tid = threadIdx.y * blockDim.x + threadIdx.x;
  const int pitch = (int)(ldx * (int64_t)sizeof(TI));                                // bytes per staged row
  int32_t* rp_s = reinterpret_cast<int32_t*>(agg_smem + (size_t)cap_rows * pitch);   // [cap_rows + 1] (+3 pad)
  int32_t* col_s = rp_s + cap_rows + 4;                                             // [4 * cap_rows] tile-local ids
  float* inv_s = reinterpret_cast<float*>(col_s + 4 * cap_rows);                    // [cap_rows] 1/(deg+1)
  const int cap_nnz = 4 * cap_rows;
  const uint32_t b32 = agg_smem_u32(&bar);
  if (tid == 0) {
    // sentences that START in [w0, w1): first sentence starting at or after w0 / w1
    const int w0 = blockIdx.x * tile_rows, w1 = w0 + tile_rows;
    // two levels of dependent loads only (see stage_window in edg_staged.cuh)
    const int a0 = w0 < N ? __ldg(row_sent + w0) : B, a1 = w1 < N ? __ldg(row_sent + w1) : B;
    const int p0 = __ldg(sent_ptr + a0), q0 = a0 < B ? __ldg(sent_ptr + a0 + 1) : p0;
    const int p1 = __ldg(sent_ptr + a1), q1 = a1 < B ? __ldg(sent_ptr + a1 + 1) : p1;
    const int r0 = (w0 < N && p0 < w0) ? q0 : p0, r1 = (w1 < N && p1 < w1) ? q1 : p1;
    range[0] = r0; range[1] = r1;
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(b32));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    const int n = r1 - r0;
    if (n > 0 && n <= cap_rows) {
      const uint32_t bytes = (uint32_t)n * (uint32_t)pitch;
      asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(b32), "r"(bytes) : "memory");
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                   ::"r"(agg_smem_u32(agg_smem)), "l"(x + (int64_t)r0 * ldx), "r"(bytes), "r"(b32) : "memory");
    }
  }
  __syncthreads();
  const int r0 = range[0], r1 = range[1], n = r1 - r0;
  if (n <= 0) return;
  if (n > cap_rows) {                               // nothing was staged
    aggregate_rows_global<TI, TO, MODE>(x, ldx, y, ldy, r0, r1, row_ptr, col);
    return;
  }
  // the tile's slice of the CSR (as tile-local ids) and 1/(deg+1) go to shared memory while the bulk copy flies
  for (int i = tid; i <= n; i += nthreads) rp_s[i] = __ldg(row_ptr + r0 + i);
  __syncthreads();
  const int e0 = rp_s[0], nnz = rp_s[n] - e0;
  const bool fits = nnz <= cap_nnz;
  if (fits)
    for (int i = tid; i < nnz; i += nthreads) col_s[i] = __ldg(col + e0 + i) - r0;
  for (int i = tid; i < n; i += nthreads) inv_s[i] = __frcp_rn((float)(rp_s[i + 1] - rp_s[i] + 1));
  __syncthreads();
  {
    uint32_t ok = 0;
    while (!ok) {
      asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                   : "=r"(ok) : "r"(b32) : "memory");
    }
  }
  if (!fits) {                                      // dense-ish graph: keep the staged copy unused, gather from global
    aggregate_rows_global<TI, TO, MODE>(x, ldx, y, ldy, r0, r1, row_ptr, col);
    return;
  }
  // ---- hot loop: shared memory only -------------------------------------------------------------------
  const uint32_t xs = agg_smem_u32(agg_smem) + threadIdx.x * 16;     // this thread's 16-byte column of the window
  TO* yrow = y + (int64_t)(r0 + (int)threadIdx.y) * ldy + threadIdx.x * E;
  const int64_t ystep = (int64_t)blockDim.y * ldy;
  for (int lr = threadIdx.y; lr < n; lr += blockDim.y, yrow += ystep) {
    const int beg = rp_s[lr] - e0, end = rp_s[lr + 1] - e0;
    float acc[E];
#pragma unroll
    for (int k = 0; k < E; ++k) acc[k] = 0.f;
#pragma unroll 2
    for (int e = beg; e < end; ++e) {
      const int j = col_s[e];
      uint32_t w0, w1, w2, w3;
      asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(w0), "=r"(w1), "=r"(w2), "=r"(w3) : "r"(xs + (uint32_t)(j * pitch)));
      if (sizeof(TI) == 2 && MODE == 0) {              // plain sum of bf16 rows: one mixed-precision add per element
        add_bf16x2(w0, acc[0], acc[1]); add_bf16x2(w1, acc[2], acc[3]);
        add_bf16x2(w2, acc[4], acc[5]); add_bf16x2(w3, acc[6], acc[7]);
        continue;
      }
      float v[8];
      if (sizeof(TI) == 2) {
        v[0] = __uint_as_float(w0 << 16); v[1] = __uint_as_float(w0 & 0xffff0000u);
        v[2] = __uint_as_float(w1 << 16); v[3] = __uint_as_float(w1 & 0xffff0000u);
        v[4] = __uint_as_float(w2 << 16); v[5] = __uint_as_float(w2 & 0xffff0000u);
        v[6] = __uint_as_float(w3 << 16); v[7] = __uint_as_float(w3 & 0xffff0000u);
      } else {
        v[0] = __uint_as_float(w0); v[1] = __uint_as_float(w1); v[2] = __uint_as_float(w2); v[3] = __uint_as_float(w3);
      }
      if (MODE == 1) {
        const float wgt = inv_s[j];
#pragma unroll
        for (int k = 0; k < E; ++k) acc[k] = fmaf(v[k], wgt, acc[k]);
      } else {
#pragma unroll
        for (int k = 0; k < E; ++k) acc[k] += v[k];
      }
    }
    if (MODE == 0) {
      const float inv = inv_s[lr];                 // 1 / (rowsum(adj) + 1), gcn.py:35
#pragma unroll
      for (int k = 0; k < E; ++k) acc[k] *= inv;
    }
    store_chunk<TO, E>(yrow, acc);
  }
}

template <typename TI, typename TO>
static int launch_aggregate(const void* x, int64_t ldx, void* y, int64_t ldy, int N, int D,
                            const int32_t* row_ptr, const int32_t* col, int mode, const int32_t* sent_ptr,
                            const int32_t* row_sent, int B, int max_len, cudaStream_t s) {
  constexpr int E = Vec16<TI>::kElems;
  const int chunks = (D + E - 1) / E;
  if (ldx < (int64_t)chunks * E || ldy < (int64_t)chunks * E) return EDG_ERR_ALIGN;
  if (chunks > 256) return EDG_ERR_UNSUPPORTED;
  const size_t pitch = (size_t)ldx * sizeof(TI);
  // staged variant: ~72 KB windows (3 blocks per SM); falls back to the flat kernel when a
  // sentence cannot fit next to a useful window
  int cap_rows = (int)((72 * 1024) / (pitch + 32));
  int tile_rows = cap_rows - max_len + 1;
  int max_threads = 384;        // 3 blocks x 380 threads per SM: 40.6 / 39.6 us at C2 (256 threads: 43.9 / 43.0, 512: 46.4 / 45.7)
  if (tile_rows < 16) {
    // long sentences (config 5: up to 200 tokens): one ~200 KB window per SM, so the block itself must bring
    // the warps that hide the shared-memory latency (256 threads alone reached 34 % of the HBM peak)
    cap_rows = (int)((200 * 1024) / (pitch + 32));
    tile_rows = cap_rows - max_len + 1;
    max_threads = 1024;
  }
  const bool staged = sent_ptr && row_sent && B > 0 && max_len > 0 && tile_rows >= 8;
  if (!staged) {
    const int64_t total = (int64_t)N * chunks;
    const unsigned blocks = (unsigned)((total + 255) / 256);
    if (mode == 0) aggregate_flat_kernel<TI, TO, 0><<<blocks, 256, 0, s>>>((const TI*)x, ldx, (TO*)y, ldy, N, chunks, row_ptr, col);
    else aggregate_flat_kernel<TI, TO, 1><<<blocks, 256, 0, s>>>((const TI*)x, ldx, (TO*)y, ldy, N, chunks, row_ptr, col);
    return check_launch();
  }
  int rpb = max_threads / chunks;
  if (rpb > 32) rpb = 32;
  if (rpb < 1) rpb = 1;
  dim3 block(chunks, rpb);
  const size_t smem = (size_t)cap_rows * pitch + (size_t)(6 * cap_rows + 8) * sizeof(int32_t);
  const unsigned blocks = (unsigned)((N + tile_rows - 1) / tile_rows);
  // two instantiations per mode: <= 384-thread and <= 1024-thread blocks
  const bool big = max_threads > 384;
  void (*kern)(const TI*, int64_t, TO*, int64_t, int, int, int, int, const int32_t*, const int32_t*, const int32_t*,
               const int32_t*);
  if (mode == 0) kern = big ? aggregate_staged_kernel<TI, TO, 0, 1024> : aggregate_staged_kernel<TI, TO, 0, 384>;
  else kern = big ? aggregate_staged_kernel<TI, TO, 1, 1024> : aggregate_staged_kernel<TI, TO, 1, 384>;
  if (int rc_ = ensure_dyn_smem((const void*)kern, smem)) return rc_;
  kern<<<blocks, block, smem, s>>>((const TI*)x, ldx, (TO*)y, ldy, N, B, tile_rows, cap_rows, sent_ptr, row_sent, row_ptr, col);
  return check_launch();
}

}  // namespace edg

using namespace edg;

extern "C" int edg_aggregate(const void* x, int x_dtype, int64_t ldx, void* y, int y_dtype, int64_t ldy,
                             int32_t N, int32_t D, const int32_t* row_ptr, const int32_t* col, int mode,
                             const int32_t* sent_ptr, const int32_t* row_sent, int32_t B, int32_t max_len,
                             edg_stream stream) {
  if (N < 0 || D <= 0 || (mode != 0 && mode != 1)) return EDG_ERR_ARG;
  if (N == 0) return EDG_OK;
  if (!x || !y || !row_ptr || !col) return EDG_ERR_ARG;
  if (!aligned16(x) || !aligned16(y) || !row_pitch_ok(x_dtype, ldx) || !row_pitch_ok(y_dtype, ldy)) return EDG_ERR_ALIGN;
  cudaStream_t s = (cudaStream_t)stream;
  if (x_dtype == EDG_BF16 && y_dtype == EDG_BF16) return launch_aggregate<__nv_bfloat16, __nv_bfloat16>(x, ldx, y, ldy, N, D, row_ptr, col, mode, sent_ptr, row_sent, B, max_len, s);
  if (x_dtype == EDG_F32 && y_dtype == EDG_F32) return launch_aggregate<float, float>(x, ldx, y, ldy, N, D, row_ptr, col, mode, sent_ptr, row_sent, B, max_len, s);
  if (x_dtype == EDG_F32 && y_dtype == EDG_BF16) return launch_aggregate<float, __nv_bfloat16>(x, ldx, y, ldy, N, D, row_ptr, col, mode, sent_ptr, row_sent, B, max_len, s);
  if (x_dtype == EDG_BF16 && y_dtype == EDG_F32) return launch_aggregate<__nv_bfloat16, float>(x, ldx, y, ldy, N, D, row_ptr, col, mode, sent_ptr, row_sent, B, max_len, s);
  return EDG_ERR_DTYPE;
}
