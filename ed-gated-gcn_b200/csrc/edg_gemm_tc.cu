// tcgen05 (5th-gen tensor core) GEMMs for the bf16 mode -- sm_100a only.
//
//   linear_tc : C[M,Nout] = act(A[M,K] * W[Nout,K]^T + bias)     (K-major A and B, TMA-fed)
//   wgrad_tc  : P[s][K1,K2] = A[rows_s,K1]^T * B[rows_s,K2]       (MN-major A and B, split over rows)
//
// Structure of both (one CTA per SM, 192 threads):
//   warp 0      : TMA producer   (cp.async.bulk.tensor -> 128B-swizzled smem ring, mbarrier tx)
//   warp 1      : TMEM allocator + single-thread tcgen05.mma issuer (accumulators in TMEM)
//   warps 2..5  : epilogue       (tcgen05.ld -> bias/activation -> global), one TMEM lane quarter each
// linear_tc is persistent over (m,n) tiles with two TMEM accumulator stages, so the epilogue
// of tile i overlaps the MMAs of tile i+1.
#include <cuda.h>
#include <string.h>

#include "edg_common.cuh"

namespace edg {

// ---------------------------------------------------------------------------------------------
// PTX wrappers
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ uint32_t mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok;
}
// Bounded wait: a protocol bug traps instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++spins > (1u << 22)) __trap();
  }
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
// TMA load delivered to the same shared-memory offset (and mbarrier) of every CTA in `cta_mask` of the cluster
__device__ __forceinline__ void tma_load_2d_mc(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1, uint16_t cta_mask) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%4, %5}], [%2], %3;"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "h"(cta_mask), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(map)) : "memory");
}

__device__ __forceinline__ void tmem_alloc(uint32_t dst_smem, uint32_t cols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(cols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t cols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
// D[tmem] (+)= A[smem desc] * B[smem desc], bf16 inputs, fp32 accumulate; issued by ONE thread.
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// mbarrier arrives once every MMA issued so far by this thread has completed.
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// the same, arriving on the barrier at this offset in every CTA of `cta_mask`
__device__ __forceinline__ void umma_commit_mc(uint32_t bar, uint16_t cta_mask) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(bar), "h"(cta_mask) : "memory");
}
// 32 lanes x 32 consecutive fp32 columns: thread `lane` gets row (lane quarter base + lane).
__device__ __forceinline__ void tmem_ld_32x32_nowait(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// Shared-memory matrix descriptor (cute::UMMA::SmemDescriptor, sm100 version = 1):
//   [0,14) start>>4 | [16,30) leading byte offset>>4 | [32,46) stride byte offset>>4 |
//   [46,48) version=1 | [61,64) layout (2 = SWIZZLE_128B)
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes, uint32_t layout) {
  uint64_t d = 0;                                 // layout: 2 = SWIZZLE_128B, 4 = SWIZZLE_64B
  d |= (uint64_t)((saddr & 0x3ffffu) >> 4);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3fffu) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3fffu) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)layout << 61;
  return d;
}
__device__ __forceinline__ uint64_t make_desc_sw128(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3ffffu) >> 4);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3fffu) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3fffu) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}

// Instruction descriptor (cute::UMMA::InstrDescriptor), kind::f16, bf16 x bf16 (or fp16 x fp16) -> fp32.
static inline uint32_t make_idesc_bf16(int M, int N, int a_mn_major, int b_mn_major, bool f16 = false) {
  uint32_t d = 0;
  d |= 1u << 4;                         // c_format  = F32
  d |= (f16 ? 0u : 1u) << 7;            // a_format  = BF16 (1) / F16 (0)
  d |= (f16 ? 0u : 1u) << 10;           // b_format  = BF16 (1) / F16 (0)
  d |= (uint32_t)(a_mn_major & 1) << 15;
  d |= (uint32_t)(b_mn_major & 1) << 16;
  d |= (uint32_t)(N >> 3) << 17;
  d |= (uint32_t)(M >> 4) << 24;
  return d;
}

// 1.0 in the operand format the instruction descriptor names (bf16 0x3F80, fp16 0x3C00)
__device__ __forceinline__ uint16_t one_of(uint32_t idesc) { return ((idesc >> 7) & 7u) ? (uint16_t)0x3F80 : (uint16_t)0x3C00; }

// ---------------------------------------------------------------------------------------------
// common tile constants
// ---------------------------------------------------------------------------------------------
constexpr int kBlockM = 128;
constexpr int kBlockK = 64;                       // 64 bf16 = one 128-byte swizzle row
constexpr int kStages = 4;
constexpr int kABytes = kBlockM * kBlockK * 2;    // 16 KB
constexpr int kBBytesMax = 256 * kBlockK * 2;     // 32 KB
constexpr int kStageBytes = kABytes + kBBytesMax; // 48 KB
constexpr int kTmemCols = 512;
constexpr int kAccStride = 256;                   // TMEM columns per accumulator stage
constexpr int kThreads = 192;          // wgrad: TMA warp, MMA warp, 4 epilogue warps
constexpr int kLinThreads = 320;       // linear: TMA warp, MMA warp, 8 epilogue warps (2 per TMEM lane quarter)
constexpr int kMaxBias = 1024;
constexpr size_t kSmemBytes = 1024 + (size_t)kStages * kStageBytes + kMaxBias * sizeof(float) + 256;

struct SmemLayout {
  uint32_t base;       // 1024-aligned shared address of stage 0
  __device__ uint32_t a(int s) const { return base + s * kStageBytes; }
  __device__ uint32_t b(int s) const { return base + s * kStageBytes + kABytes; }
  __device__ uint32_t bias() const { return base + kStages * kStageBytes; }
  __device__ uint32_t bars() const { return bias() + kMaxBias * sizeof(float); }
  __device__ uint32_t full(int s) const { return bars() + 8 * s; }
  __device__ uint32_t empty(int s) const { return bars() + 8 * (kStages + s); }
  __device__ uint32_t tfull(int s) const { return bars() + 8 * (2 * kStages + s); }
  __device__ uint32_t tempty(int s) const { return bars() + 8 * (2 * kStages + 2 + s); }
  __device__ uint32_t tmem_slot() const { return bars() + 8 * (2 * kStages + 4); }
};

template <typename TC> struct OutVec;
template <> struct OutVec<float> {
  static constexpr int G = 4;
  __device__ static __forceinline__ void store(float* p, const float* v) { *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]); }
};
template <> struct OutVec<__nv_bfloat16> {
  static constexpr int G = 8;
  __device__ static __forceinline__ void store(__nv_bfloat16* p, const float* v) {
    uint32_t w[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      __nv_bfloat162 h = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
      w[i] = *reinterpret_cast<uint32_t*>(&h);
    }
    *reinterpret_cast<uint4*>(p) = make_uint4(w[0], w[1], w[2], w[3]);
  }
};

// ---------------------------------------------------------------------------------------------
// linear_tc
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float apply_act(float x, int act) {
  if (act == EDG_ACT_SIGMOID) return __fdividef(1.0f, 1.0f + __expf(-x));
  if (act == EDG_ACT_RELU) return fmaxf(x, 0.f);
  return x;
}

// one 32-column chunk of one accumulator row -> bias, activation, convert, 128-bit stores
template <typename TC>
__device__ __forceinline__ void epilogue_chunk(const uint32_t (&r)[32], int col0, int Nout, int64_t ldc, int act,
                                               const float* __restrict__ bias_s, TC* __restrict__ crow) {
  constexpr int G = OutVec<TC>::G;
  if (col0 + 32 <= Nout) {                      // interior chunk: no per-element guards
#pragma unroll
    for (int g = 0; g < 32; g += G) {
      float v[G];
#pragma unroll
      for (int j = 0; j < G; ++j) v[j] = apply_act(__uint_as_float(r[g + j]) + bias_s[col0 + g + j], act);
      OutVec<TC>::store(crow + col0 + g, v);
    }
  } else {                                      // last chunk of the row: zero the padding, skip what is past ldc
#pragma unroll
    for (int g = 0; g < 32; g += G) {
      const int col = col0 + g;
      if (col + G <= ldc) {
        float v[G];
#pragma unroll
        for (int j = 0; j < G; ++j) {
          const int cj = col + j;
          v[j] = (cj < Nout) ? apply_act(__uint_as_float(r[g + j]) + bias_s[cj < kMaxBias ? cj : 0], act) : 0.f;
        }
        OutVec<TC>::store(crow + col, v);
      }
    }
  }
}

template <typename TC>
__global__ void __launch_bounds__(kLinThreads, 1)
linear_tc_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_w,
                 int M, int K, int Nout, int block_n, int n_tiles, int num_tiles, uint32_t idesc,
                 const float* __restrict__ bias, int act, TC* __restrict__ C, int64_t ldc) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  SmemLayout L;
  L.base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int num_kb = (K + kBlockK - 1) / kBlockK;
  float* bias_s = reinterpret_cast<float*>(smem_raw + (L.bias() - smem_u32(smem_raw)));

  for (int i = threadIdx.x; i < kMaxBias; i += kLinThreads) bias_s[i] = (bias && i < Nout) ? bias[i] : 0.f;
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&map_a);
    tma_prefetch_desc(&map_w);
    for (int s = 0; s < kStages; ++s) { mbar_init(L.full(s), 1); mbar_init(L.empty(s), 1); }
    for (int s = 0; s < 2; ++s) { mbar_init(L.tfull(s), 1); mbar_init(L.tempty(s), 8); }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(L.tmem_slot(), kTmemCols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tmem_base) : "r"(L.tmem_slot()));

  if (warp == 0) {
    if (lane == 0) {
      const uint32_t stage_tx = kABytes + (uint32_t)block_n * kBlockK * 2;
      int stage = 0; uint32_t phase = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        const int m0 = (tile / n_tiles) * kBlockM, n0 = (tile % n_tiles) * block_n;
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(L.empty(stage), phase ^ 1);
          mbar_expect_tx(L.full(stage), stage_tx);
          tma_load_2d(L.a(stage), &map_a, L.full(stage), kb * kBlockK, m0);
          tma_load_2d(L.b(stage), &map_w, L.full(stage), kb * kBlockK, n0);
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      int stage = 0; uint32_t phase = 0;
      int it = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++it) {
        const int as = it & 1;
        const uint32_t aphase = (it >> 1) & 1;
        mbar_wait(L.tempty(as), aphase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + as * kAccStride;
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(L.full(stage), phase);
          tc_fence_after();
#pragma unroll
          for (int k = 0; k < kBlockK / 16; ++k) {
            const uint64_t ad = make_desc_sw128(L.a(stage) + k * 32, 16, 1024);
            const uint64_t bd = make_desc_sw128(L.b(stage) + k * 32, 16, 1024);
            umma_bf16(d_tmem, ad, bd, idesc, (kb | k) != 0);
          }
          umma_commit(L.empty(stage));           // frees the smem slot when these MMAs retire
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
        umma_commit(L.tfull(as));                // accumulator ready for the epilogue
      }
    }
  } else {
    // 8 epilogue warps: warp w reads TMEM lane quarter (w & 3); the two warps of a quarter take alternate
    // 32-column chunks.  TMEM loads are software-pipelined one chunk ahead of the arithmetic.
    const int q = warp & 3;
    const int half = (warp - 2) >> 2;
    const int n_chunks = (block_n + 31) / 32;
    int it = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++it) {
      const int as = it & 1;
      const uint32_t aphase = (it >> 1) & 1;
      const int m0 = (tile / n_tiles) * kBlockM, n0 = (tile % n_tiles) * block_n;
      mbar_wait(L.tfull(as), aphase);
      tc_fence_after();
      const int row = m0 + q * 32 + lane;
      const bool row_ok = row < M;
      TC* crow = C + (int64_t)(row_ok ? row : 0) * ldc;
      const uint32_t tbase = tmem_base + ((uint32_t)(q * 32) << 16) + as * kAccStride;
      uint32_t ra[32], rb[32];
      int ci = half;
      if (ci < n_chunks) tmem_ld_32x32_nowait(tbase + ci * 32, ra);
      while (ci < n_chunks) {
        tmem_wait_ld();
        const int nxt = ci + 2;
        if (nxt < n_chunks) tmem_ld_32x32_nowait(tbase + nxt * 32, rb);
        if (row_ok && n0 + ci * 32 < ldc) epilogue_chunk<TC>(ra, n0 + ci * 32, Nout, ldc, act, bias_s, crow);
        ci = nxt;
        if (ci >= n_chunks) break;
        tmem_wait_ld();
        const int nx2 = ci + 2;
        if (nx2 < n_chunks) tmem_ld_32x32_nowait(tbase + nx2 * 32, ra);
        if (row_ok && n0 + ci * 32 < ldc) epilogue_chunk<TC>(rb, n0 + ci * 32, Nout, ldc, act, bias_s, crow);
        ci = nx2;
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(L.tempty(as));
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, kTmemCols);
  }
}

// ---------------------------------------------------------------------------------------------
// linear_ws : the same GEMM with the WEIGHT TILE STATIONARY in shared memory.
// At D = 300 the streaming kernel above re-reads its [block_n x K] weight tile from L2 for every M tile
// (100 KB per 40 KB of output) and is L2-bandwidth bound.  Here CTA c keeps the weight rows of ONE N tile
// (c % n_tiles) resident for its whole life and walks the M tiles c / n_tiles, + gridDim/n_tiles, ...; only
// the activation tiles stream through the TMA ring.  The CTAs of the same M tile run side by side, so the
// second read of an activation tile is an L2 hit.
// ---------------------------------------------------------------------------------------------
constexpr int kWsMaxStages = 8;
constexpr int kSplitCross = 128;    // TMEM column offset of the cross-term accumulator inside one accumulator stage
struct WsLayout {
  uint32_t base; int w_bytes_kb; int num_kb; int stages; int w_boxes; int a_bytes;
  __device__ uint32_t w(int kb) const { return base + kb * w_bytes_kb; }
  __device__ uint32_t a(int s) const { return base + w_boxes * w_bytes_kb + s * a_bytes; }
  __device__ uint32_t bias() const { return a(stages); }
  __device__ uint32_t bars() const { return bias() + kMaxBias * sizeof(float); }
  __device__ uint32_t full(int s) const { return bars() + 8 * s; }
  __device__ uint32_t empty(int s) const { return bars() + 8 * (kWsMaxStages + s); }
  __device__ uint32_t tfull(int s) const { return bars() + 8 * (2 * kWsMaxStages + s); }
  __device__ uint32_t tempty(int s) const { return bars() + 8 * (2 * kWsMaxStages + 2 + s); }
  __device__ uint32_t wfull() const { return bars() + 8 * (2 * kWsMaxStages + 4); }
  __device__ uint32_t tmem_slot() const { return bars() + 8 * (2 * kWsMaxStages + 5); }
};

// Split operands (the fp32-parity mode, see edg_split.cu): an fp32 matrix x is stored as two fp16 matrices side by
// side, row = [ hi | lo ] with hi = fp16(x s), lo = fp16(x s - hi), s = split_scale(max |x|) a power of two.
// hi + lo carries 22 significant bits of x s, and  a w^T = (a_hi w_hi^T + a_hi w_lo^T + a_lo w_hi^T) / (s_a s_w)
// to ~2^-21 per product with fp32 accumulation in TMEM -- three fp16 MMAs per k step instead of one.
__device__ __forceinline__ float split_scale(float amax) {          // amax * s in [2^13, 2^14)
  const int e = (int)((__float_as_uint(amax) >> 23) & 0xffu);
  int se = 267 - e;
  se = se < 1 ? 1 : (se > 254 ? 254 : se);
  return __uint_as_float((uint32_t)se << 23);
}
__device__ __forceinline__ float split_inv_scale(float amax) {
  const int e = (int)((__float_as_uint(amax) >> 23) & 0xffu);
  int se = 267 - e;
  se = se < 1 ? 1 : (se > 254 ? 254 : se);
  return se <= 253 ? __uint_as_float((uint32_t)(254 - se) << 23) : __uint_as_float(0x00400000u);
}

// one 32-column chunk of one accumulator row of the split kernel: scale back, bias, activation, fp32 stores;
// only columns below `col_end` (what this CTA's N tile owns) are written, columns in [Nout, col_end) as zeros
__device__ __forceinline__ void epilogue_chunk_scaled(const uint32_t (&r)[32], int col0, int Nout, int col_end, int act,
                                                      float inv_a, float inv_w, const float* __restrict__ bias_s,
                                                      float* __restrict__ crow) {
#pragma unroll
  for (int g = 0; g < 32; g += 4) {
    const int col = col0 + g;
    if (col + 4 <= col_end) {
      float v[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int cj = col + j;
        v[j] = (cj < Nout) ? apply_act(__uint_as_float(r[g + j]) * inv_a * inv_w + bias_s[cj < kMaxBias ? cj : 0], act) : 0.f;
      }
      *reinterpret_cast<float4*>(crow + col) = make_float4(v[0], v[1], v[2], v[3]);
    }
  }
}

template <typename TC, bool SPLIT>
__global__ void __launch_bounds__(kLinThreads, 1)
linear_ws_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_w,
                 int M, int K, int Nout, int block_n, int n_tiles, int m_tiles, int stages, uint32_t idesc,
                 const float* __restrict__ bias, int act, TC* __restrict__ C, int64_t ldc,
                 int k_lo, const float* __restrict__ amax_a, const float* __restrict__ amax_w) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  WsLayout L;
  L.base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  L.num_kb = (K + kBlockK - 1) / kBlockK;
  L.w_bytes_kb = block_n * kBlockK * 2;
  L.stages = stages;
  L.w_boxes = SPLIT ? 2 * L.num_kb : L.num_kb;          // split: hi boxes then lo boxes
  L.a_bytes = SPLIT ? 2 * kABytes : kABytes;            // split: hi tile then lo tile
  const int num_kb = L.num_kb;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* bias_s = reinterpret_cast<float*>(smem_raw + (L.bias() - smem_u32(smem_raw)));
  const int n_tile = blockIdx.x % n_tiles, n0 = n_tile * block_n;
  const int m_first = blockIdx.x / n_tiles, m_step = gridDim.x / n_tiles;

  for (int i = threadIdx.x; i < kMaxBias; i += kLinThreads) bias_s[i] = (bias && i < Nout) ? bias[i] : 0.f;
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&map_a);
    tma_prefetch_desc(&map_w);
    for (int s = 0; s < stages; ++s) { mbar_init(L.full(s), 1); mbar_init(L.empty(s), 1); }
    for (int s = 0; s < 2; ++s) { mbar_init(L.tfull(s), 1); mbar_init(L.tempty(s), 8); }
    mbar_init(L.wfull(), 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(L.tmem_slot(), kTmemCols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tmem_base) : "r"(L.tmem_slot()));

  if (warp == 0) {
    if (lane == 0) {
      // the stationary weight tile: boxes [block_n rows x 64 k], one barrier
      mbar_expect_tx(L.wfull(), (uint32_t)(L.w_boxes * L.w_bytes_kb));
      for (int kb = 0; kb < num_kb; ++kb) tma_load_2d(L.w(kb), &map_w, L.wfull(), kb * kBlockK, n0);
      if (SPLIT)
        for (int kb = 0; kb < num_kb; ++kb) tma_load_2d(L.w(num_kb + kb), &map_w, L.wfull(), k_lo + kb * kBlockK, n0);
      int stage = 0; uint32_t phase = 0;
      for (int mt = m_first; mt < m_tiles; mt += m_step) {
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(L.empty(stage), phase ^ 1);
          mbar_expect_tx(L.full(stage), (uint32_t)L.a_bytes);
          tma_load_2d(L.a(stage), &map_a, L.full(stage), kb * kBlockK, mt * kBlockM);
          if (SPLIT) tma_load_2d(L.a(stage) + kABytes, &map_a, L.full(stage), k_lo + kb * kBlockK, mt * kBlockM);
          if (++stage == stages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      mbar_wait(L.wfull(), 0);
      int stage = 0; uint32_t phase = 0;
      int it = 0;
      for (int mt = m_first; mt < m_tiles; mt += m_step, ++it) {
        const int as = it & 1;
        const uint32_t aphase = (it >> 1) & 1;
        mbar_wait(L.tempty(as), aphase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + as * kAccStride;
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(L.full(stage), phase);
          tc_fence_after();
#pragma unroll
          for (int k = 0; k < kBlockK / 16; ++k) {
            const uint64_t ad = make_desc_sw128(L.a(stage) + k * 32, 16, 1024);
            const uint64_t bd = make_desc_sw128(L.w(kb) + k * 32, 16, 1024);
            if (SPLIT) {
              // The tensor core truncates when it accumulates, so the error grows with the length of the chain:
              // the two small products get their own accumulator (kSplitCross columns further), which keeps the
              // hi x hi chain at K/16 steps; the epilogue adds the two.
              const uint64_t al = make_desc_sw128(L.a(stage) + kABytes + k * 32, 16, 1024);
              const uint64_t bl = make_desc_sw128(L.w(num_kb + kb) + k * 32, 16, 1024);
              umma_bf16(d_tmem + kSplitCross, al, bd, idesc, (kb | k) != 0);
              umma_bf16(d_tmem + kSplitCross, ad, bl, idesc, 1);
              umma_bf16(d_tmem, ad, bd, idesc, (kb | k) != 0);
            } else {
              umma_bf16(d_tmem, ad, bd, idesc, (kb | k) != 0);
            }
          }
          umma_commit(L.empty(stage));
          if (++stage == stages) { stage = 0; phase ^= 1; }
        }
        umma_commit(L.tfull(as));
      }
    }
  } else {
    const int q = warp & 3;
    const int half = (warp - 2) >> 2;
    const int n_chunks = (block_n + 31) / 32;
    float inv_a = 1.f, inv_w = 1.f;
    int col_end = 0;
    if (SPLIT) {
      inv_a = split_inv_scale(__ldg(amax_a));
      inv_w = split_inv_scale(__ldg(amax_w));
      col_end = (n_tile == n_tiles - 1) ? (int)ldc : n0 + block_n;
      if (col_end > (int)ldc) col_end = (int)ldc;
    }
    int it = 0;
    for (int mt = m_first; mt < m_tiles; mt += m_step, ++it) {
      const int as = it & 1;
      const uint32_t aphase = (it >> 1) & 1;
      mbar_wait(L.tfull(as), aphase);
      tc_fence_after();
      const int row = mt * kBlockM + q * 32 + lane;
      const bool row_ok = row < M;
      TC* crow = C + (int64_t)(row_ok ? row : 0) * ldc;
      const uint32_t tbase = tmem_base + ((uint32_t)(q * 32) << 16) + as * kAccStride;
      uint32_t ra[32], rb[32];
      auto emit = [&](const uint32_t (&r)[32], int ci) {
        if (!row_ok) return;
        if constexpr (SPLIT) {
          epilogue_chunk_scaled(r, n0 + ci * 32, Nout, col_end, act, inv_a, inv_w, bias_s, reinterpret_cast<float*>(crow));
        } else {
          if (n0 + ci * 32 < ldc) epilogue_chunk<TC>(r, n0 + ci * 32, Nout, ldc, act, bias_s, crow);
        }
      };
      int ci = half;
      if constexpr (SPLIT) {
        for (; ci < n_chunks; ci += 2) {
          tmem_ld_32x32_nowait(tbase + ci * 32, ra);
          tmem_ld_32x32_nowait(tbase + kSplitCross + ci * 32, rb);
          tmem_wait_ld();
#pragma unroll
          for (int j = 0; j < 32; ++j) ra[j] = __float_as_uint(__uint_as_float(ra[j]) + __uint_as_float(rb[j]));
          emit(ra, ci);
        }
      }
      if (ci < n_chunks) tmem_ld_32x32_nowait(tbase + ci * 32, ra);
      while (ci < n_chunks) {
        tmem_wait_ld();
        const int nxt = ci + 2;
        if (nxt < n_chunks) tmem_ld_32x32_nowait(tbase + nxt * 32, rb);
        emit(ra, ci);
        ci = nxt;
        if (ci >= n_chunks) break;
        tmem_wait_ld();
        const int nx2 = ci + 2;
        if (nx2 < n_chunks) tmem_ld_32x32_nowait(tbase + nx2 * 32, ra);
        emit(rb, ci);
        ci = nx2;
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(L.tempty(as));
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, kTmemCols);
  }
}

// ---------------------------------------------------------------------------------------------
// wgrad_tc : both operands MN-major (rows of the activation matrices are the GEMM K dimension)
//   smem stage = 64 activation rows; A = 2 boxes [64 rows x 64 cols], B = block_n/64 such boxes.
//   canonical MN-major SWIZZLE_128B layout: 64-column atom contiguous (128 B), 8-row groups
//   1024 B apart (SBO), next 64-column atom one box (8192 B) further (LBO).
// ---------------------------------------------------------------------------------------------
constexpr int kBoxBytes = 64 * 64 * 2;   // 8 KB

// 32 consecutive fp32 of one partial-sum row: 128-bit stores when the row pitch allows, scalar otherwise
__device__ __forceinline__ void store_partial_chunk(float* __restrict__ prow, int col0, int K2e, const uint32_t (&r)[32], bool valid) {
  if ((K2e & 3) == 0 && col0 + 32 <= K2e) {
#pragma unroll
    for (int j = 0; j < 32; j += 4) {
      float4 v = valid ? make_float4(__uint_as_float(r[j]), __uint_as_float(r[j + 1]), __uint_as_float(r[j + 2]), __uint_as_float(r[j + 3]))
                       : make_float4(0.f, 0.f, 0.f, 0.f);
      *reinterpret_cast<float4*>(prow + col0 + j) = v;
    }
  } else {
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      const int col = col0 + j;
      if (col < K2e) prow[col] = valid ? __uint_as_float(r[j]) : 0.f;
    }
  }
}

// Bias gradients ride along for free: `ones_a` >= 0 plants a column of ones at A column `ones_a` (= K1), so
// output row K1 is the column sum of B; `ones_b` >= 0 does the same on the B side (output column K2 = column
// sums of A).  The ones are written into the landed smem tile (swizzled address) right before the MMAs.
__device__ __forceinline__ void plant_ones(uint32_t box_base, int col_in_box, int rows_valid, int lane, uint16_t one = 0x3F80) {
  // box = [64 rows x 64 bf16] with 128-byte rows, 16-byte chunks XOR-swizzled by (row & 7)
  const int chunk = col_in_box >> 3, within = (col_in_box & 7) * 2;
  for (int r = lane; r < 64; r += 32) {
    const uint32_t addr = box_base + r * 128 + (((chunk ^ (r & 7)) << 4) | within);
    const uint16_t v = (r < rows_valid) ? one : (uint16_t)0;   // 1.0 (bf16 0x3F80 / fp16 0x3C00) for real rows only
    asm volatile("st.shared.u16 [%0], %1;" ::"r"(addr), "h"(v) : "memory");
  }
}

// body shared by the single-problem kernel and the batched one (`split` = row range, `slot` = partial-sum slab)
__device__ __forceinline__ void wgrad_tc_body(const CUtensorMap& map_a, const CUtensorMap& map_b, int split, int slot,
                                              int R, int K1e, int K2e, int block_n, int rows_per, uint32_t idesc,
                                              int ones_a, int ones_b, float* __restrict__ partial) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  SmemLayout L;
  L.base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m0 = blockIdx.x * kBlockM, n0 = blockIdx.y * block_n;
  const int r_beg = split * rows_per;
  const int r_end = min(R, r_beg + rows_per);
  const int num_kb = (r_end > r_beg) ? (r_end - r_beg + kBlockK - 1) / kBlockK : 0;
  const int n_boxes = block_n / 64;
  const bool plant_a = ones_a >= m0 && ones_a < m0 + kBlockM;
  const bool plant_b = ones_b >= n0 && ones_b < n0 + block_n;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&map_a);
    tma_prefetch_desc(&map_b);
    for (int s = 0; s < kStages; ++s) { mbar_init(L.full(s), 1); mbar_init(L.empty(s), 1); }
    mbar_init(L.tfull(0), 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(L.tmem_slot(), 256);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tmem_base) : "r"(L.tmem_slot()));

  if (warp == 0) {
    if (lane == 0) {
      const uint32_t stage_tx = (uint32_t)(2 + n_boxes) * kBoxBytes;
      int stage = 0; uint32_t phase = 0;
      for (int kb = 0; kb < num_kb; ++kb) {
        mbar_wait(L.empty(stage), phase ^ 1);
        mbar_expect_tx(L.full(stage), stage_tx);
        const int r0 = r_beg + kb * kBlockK;
        tma_load_2d(L.a(stage), &map_a, L.full(stage), m0, r0);
        tma_load_2d(L.a(stage) + kBoxBytes, &map_a, L.full(stage), m0 + 64, r0);
        for (int j = 0; j < n_boxes; ++j)
          tma_load_2d(L.b(stage) + j * kBoxBytes, &map_b, L.full(stage), n0 + 64 * j, r0);
        if (++stage == kStages) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1) {
    int stage = 0; uint32_t phase = 0;
    for (int kb = 0; kb < num_kb; ++kb) {
      mbar_wait(L.full(stage), phase);
      if (plant_a || plant_b) {                      // whole warp: ones column into the landed tile
        const int rows_valid = r_end - (r_beg + kb * kBlockK);
        if (plant_a) plant_ones(L.a(stage) + ((ones_a - m0) >> 6) * kBoxBytes, (ones_a - m0) & 63, rows_valid, lane, one_of(idesc));
        if (plant_b) plant_ones(L.b(stage) + ((ones_b - n0) >> 6) * kBoxBytes, (ones_b - n0) & 63, rows_valid, lane, one_of(idesc));
        fence_proxy_async();                         // generic-proxy writes -> visible to the tensor core (async proxy)
        __syncwarp();
      }
      tc_fence_after();
      if (lane == 0) {
#pragma unroll
        for (int k = 0; k < kBlockK / 16; ++k) {
          const uint64_t ad = make_desc_sw128(L.a(stage) + k * 2048, kBoxBytes, 1024);
          const uint64_t bd = make_desc_sw128(L.b(stage) + k * 2048, kBoxBytes, 1024);
          umma_bf16(tmem_base, ad, bd, idesc, (kb | k) != 0);
        }
        umma_commit(L.empty(stage));
      }
      __syncwarp();
      if (++stage == kStages) { stage = 0; phase ^= 1; }
    }
    if (lane == 0) umma_commit(L.tfull(0));
  } else {
    const int q = warp & 3;
    float* P = partial + (int64_t)slot * K1e * K2e;
    const int row = m0 + q * 32 + lane;
    if (num_kb > 0) {
      mbar_wait(L.tfull(0), 0);
      tc_fence_after();
    }
    for (int c0 = 0; c0 < block_n; c0 += 32) {
      uint32_t r[32];
      if (num_kb > 0) { tmem_ld_32x32_nowait(tmem_base + ((uint32_t)(q * 32) << 16) + c0, r); tmem_wait_ld(); }
      if (row < K1e) store_partial_chunk(P + (int64_t)row * K2e, n0 + c0, K2e, r, num_kb > 0);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 256);
  }
}

__global__ void __launch_bounds__(kThreads, 1)
wgrad_tc_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
                int R, int K1e, int K2e, int block_n, int rows_per, uint32_t idesc, int ones_a, int ones_b,
                float* __restrict__ partial) {
  wgrad_tc_body(map_a, map_b, blockIdx.z, blockIdx.z, R, K1e, K2e, block_n, rows_per, idesc, ones_a, ones_b, partial);
}

// Several same-shaped weight gradients in ONE launch (the Linears of the gate MLPs: 4 problems of
// [D x B] x [B x D] at C2): blockIdx.z = problem * splits + split; slab z of `partial` is problem-major.
constexpr int kWgradBatchMax = 8;
struct WgradBatchMaps {
  CUtensorMap a[kWgradBatchMax];
  CUtensorMap b[kWgradBatchMax];
};
__global__ void __launch_bounds__(kThreads, 1)
wgrad_tc_batch_kernel(const __grid_constant__ WgradBatchMaps maps, int splits, int R, int K1e, int K2e, int block_n,
                      int rows_per, uint32_t idesc, int ones_a, int ones_b, float* __restrict__ partial) {
  const int p = blockIdx.z / splits, split = blockIdx.z - p * splits;
  wgrad_tc_body(maps.a[p], maps.b[p], split, blockIdx.z, R, K1e, K2e, block_n, rows_per, idesc, ones_a, ones_b, partial);
}

// ---------------------------------------------------------------------------------------------
// wgrad_tall : one CTA owns ALL M tiles (K1 <= 384) of one N tile (<= 160 columns) for its row range, so the
// A operand (K1 columns) is read once per N tile and the B operand once overall: 210 MB of L2->SM traffic
// at C2 instead of 343 MB for the [128 x 192] tiles of wgrad_tc (which is L2-bandwidth bound).
//   stage (64 rows): A = 2*m_tiles boxes [64 rows x 64 cols] SW128, B = block_n/32 boxes [64 rows x 32 cols] SW64
//   TMEM: accumulator of M tile mt at columns mt*block_n (m_tiles*block_n <= 512)
// ---------------------------------------------------------------------------------------------
constexpr int kTallStages = 3;
constexpr int kTallMaxM = 3;
constexpr int kTallABytes = kTallMaxM * 2 * kBoxBytes;       // 48 KB
constexpr int kTallBBox = 64 * 32 * 2;                       // 4 KB
constexpr int kTallBBytes = 5 * kTallBBox;                   // 20 KB (block_n <= 160)
constexpr int kTallStageBytes = kTallABytes + kTallBBytes;   // 68 KB
constexpr size_t kTallSmem = 1024 + (size_t)kTallStages * kTallStageBytes + 256;

__device__ __forceinline__ void plant_ones_sw64(uint32_t box_base, int col_in_box, int rows_valid, int lane, uint16_t one = 0x3F80) {
  // box = [64 rows x 32 bf16] with 64-byte rows, 16-byte chunks XOR-swizzled by ((row >> 1) & 3)
  const int chunk = col_in_box >> 3, within = (col_in_box & 7) * 2;
  for (int r = lane; r < 64; r += 32) {
    const uint32_t addr = box_base + r * 64 + (((chunk ^ ((r >> 1) & 3)) << 4) | within);
    const uint16_t v = (r < rows_valid) ? one : (uint16_t)0;
    asm volatile("st.shared.u16 [%0], %1;" ::"r"(addr), "h"(v) : "memory");
  }
}

__global__ void __launch_bounds__(kThreads, 1)
wgrad_tall_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
                  int R, int K1e, int K2e, int m_tiles, int block_n, int rows_per, uint32_t idesc, int ones_a, int ones_b,
                  float* __restrict__ partial) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  auto sa = [&](int st) { return base + st * kTallStageBytes; };
  auto sb = [&](int st) { return base + st * kTallStageBytes + kTallABytes; };
  const uint32_t bars = base + kTallStages * kTallStageBytes;
  auto full = [&](int st) { return bars + 8 * st; };
  auto empty = [&](int st) { return bars + 8 * (kTallStages + st); };
  const uint32_t tfull = bars + 8 * (2 * kTallStages);
  const uint32_t tmem_slot = bars + 8 * (2 * kTallStages + 1);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n0 = blockIdx.x * block_n;
  const int r_beg = blockIdx.y * rows_per;
  const int r_end = min(R, r_beg + rows_per);
  const int num_kb = (r_end > r_beg) ? (r_end - r_beg + kBlockK - 1) / kBlockK : 0;
  const int a_boxes = 2 * m_tiles, b_boxes = block_n / 32;
  const bool plant_a = ones_a >= 0;
  const bool plant_b = ones_b >= n0 && ones_b < n0 + block_n;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&map_a);
    tma_prefetch_desc(&map_b);
    for (int s = 0; s < kTallStages; ++s) { mbar_init(full(s), 1); mbar_init(empty(s), 1); }
    mbar_init(tfull, 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, kTmemCols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));

  if (warp == 0) {
    if (lane == 0) {
      const uint32_t stage_tx = (uint32_t)a_boxes * kBoxBytes + (uint32_t)b_boxes * kTallBBox;
      int stage = 0; uint32_t phase = 0;
      for (int kb = 0; kb < num_kb; ++kb) {
        mbar_wait(empty(stage), phase ^ 1);
        mbar_expect_tx(full(stage), stage_tx);
        const int r0 = r_beg + kb * kBlockK;
        for (int j = 0; j < a_boxes; ++j) tma_load_2d(sa(stage) + j * kBoxBytes, &map_a, full(stage), 64 * j, r0);
        for (int j = 0; j < b_boxes; ++j) tma_load_2d(sb(stage) + j * kTallBBox, &map_b, full(stage), n0 + 32 * j, r0);
        if (++stage == kTallStages) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1) {
    int stage = 0; uint32_t phase = 0;
    for (int kb = 0; kb < num_kb; ++kb) {
      mbar_wait(full(stage), phase);
      if (plant_a || plant_b) {
        const int rows_valid = r_end - (r_beg + kb * kBlockK);
        if (plant_a) plant_ones(sa(stage) + (ones_a >> 6) * kBoxBytes, ones_a & 63, rows_valid, lane, one_of(idesc));
        if (plant_b) plant_ones_sw64(sb(stage) + ((ones_b - n0) >> 5) * kTallBBox, (ones_b - n0) & 31, rows_valid, lane, one_of(idesc));
        fence_proxy_async();
        __syncwarp();
      }
      tc_fence_after();
      if (lane == 0) {
#pragma unroll
        for (int k = 0; k < kBlockK / 16; ++k) {
          const uint64_t bd = make_desc(sb(stage) + k * 1024, kTallBBox, 512, 4);
          for (int mt = 0; mt < m_tiles; ++mt) {
            const uint64_t ad = make_desc(sa(stage) + mt * 2 * kBoxBytes + k * 2048, kBoxBytes, 1024, 2);
            umma_bf16(tmem_base + mt * block_n, ad, bd, idesc, (kb | k) != 0);
          }
        }
        umma_commit(empty(stage));
      }
      __syncwarp();
      if (++stage == kTallStages) { stage = 0; phase ^= 1; }
    }
    if (lane == 0) umma_commit(tfull);
  } else {
    const int q = warp & 3;
    float* P = partial + (int64_t)blockIdx.y * K1e * K2e;
    if (num_kb > 0) {
      mbar_wait(tfull, 0);
      tc_fence_after();
    }
    for (int mt = 0; mt < m_tiles; ++mt) {
      const int row = mt * kBlockM + q * 32 + lane;
      for (int c0 = 0; c0 < block_n; c0 += 32) {
        uint32_t r[32];
        if (num_kb > 0) { tmem_ld_32x32_nowait(tmem_base + ((uint32_t)(q * 32) << 16) + mt * block_n + c0, r); tmem_wait_ld(); }
        if (row < K1e) store_partial_chunk(P + (int64_t)row * K2e, n0 + c0, K2e, r, num_kb > 0);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, kTmemCols);
  }
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;      // resolved once; the pointer is process-wide and immutable
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)p;
  }
  return fn;
}

// 2-D bf16 row-major [rows, cols] (pitch ld elements), box = [box_rows, box_cols], 128B swizzle, OOB -> 0
static int make_map_bf16(CUtensorMap* map, const void* ptr, int64_t rows, int64_t cols, int64_t ld, int box_cols,
                         int box_rows, bool swizzle64 = false) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) return EDG_ERR_CUDA;
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)ld * 2};
  cuuint32_t box[2] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? EDG_OK : EDG_ERR_CUDA;
}

static int pick_block_n(int Nout, int granule, int* n_tiles) {
  int nt = (Nout + 255) / 256;
  int bn = (Nout + nt - 1) / nt;
  bn = ((bn + granule - 1) / granule) * granule;
  if (bn > 256) { ++nt; bn = (((Nout + nt - 1) / nt) + granule - 1) / granule * granule; }
  *n_tiles = (Nout + bn - 1) / bn;
  return bn;
}

template <typename TC>
static int launch_linear_tc_t(const CUtensorMap& ma, const CUtensorMap& mw, int M, int K, int Nout, int block_n,
                              int n_tiles, const float* bias, int act, void* C, int64_t ldc, cudaStream_t s) {
  if (int rc_ = ensure_dyn_smem((const void*)linear_tc_kernel<TC>, kSmemBytes)) return rc_;
  const int m_tiles = (M + kBlockM - 1) / kBlockM;
  const int num_tiles = m_tiles * n_tiles;
  const int grid = num_tiles < kNumSMs ? num_tiles : kNumSMs;
  const uint32_t idesc = make_idesc_bf16(kBlockM, block_n, 0, 0);
  linear_tc_kernel<TC><<<grid, kLinThreads, kSmemBytes, s>>>(ma, mw, M, K, Nout, block_n, n_tiles, num_tiles, idesc,
                                                          bias, act, (TC*)C, ldc);
  return check_launch();
}

// SMs the persistent projection kernel may occupy (edg_set_sm_budget): a caller that wants a collective to run NEXT to
// it leaves a few SMs free -- a one-CTA-per-SM kernel with a static tile assignment is otherwise delayed by whatever
// holds one of its SMs
static int g_sm_budget = kNumSMs;
int set_sm_budget(int n) {
  const int prev = g_sm_budget;
  g_sm_budget = n < 1 ? 1 : (n > kNumSMs ? kNumSMs : n);
  return prev;
}

template <typename TC>
static int launch_linear_ws_t(const CUtensorMap& ma, const CUtensorMap& mw, int M, int K, int Nout, int block_n,
                              int n_tiles, int stages, size_t smem, const float* bias, int act, void* C, int64_t ldc,
                              cudaStream_t s) {
  if (int rc_ = ensure_dyn_smem((const void*)linear_ws_kernel<TC, false>, 227 * 1024)) return rc_;
  const int m_tiles = (M + kBlockM - 1) / kBlockM;
  int groups = g_sm_budget / n_tiles;             // CTAs per N tile
  if (groups < 1) groups = 1;
  if (groups > m_tiles) groups = m_tiles;
  const uint32_t idesc = make_idesc_bf16(kBlockM, block_n, 0, 0);
  linear_ws_kernel<TC, false><<<groups * n_tiles, kLinThreads, smem, s>>>(ma, mw, M, K, Nout, block_n, n_tiles, m_tiles,
                                                                           stages, idesc, bias, act, (TC*)C, ldc, 0, nullptr,
                                                                           nullptr);
  return check_launch();
}

// ---- split operands (fp32-parity mode): rows = [hi | lo] fp16, lo at column k_lo = ld / 2 ----
// N tile: the widest multiple of 16 whose hi+lo weight boxes leave room for two (hi+lo) activation stages
struct SplitPlan { bool ok; int block_n, n_tiles, stages; size_t smem; };
static SplitPlan plan_linear_split(int K, int Nout) {
  SplitPlan p{};
  const int num_kb = (K + kBlockK - 1) / kBlockK;
  const size_t fixed = 1024 + kMaxBias * sizeof(float) + 512;
  const size_t budget = 227 * 1024;
  int bn = 256;
  while (bn >= 16 && fixed + (size_t)2 * num_kb * bn * kBlockK * 2 + 2 * (size_t)(2 * kABytes) > budget) bn -= 16;
  if (bn > kSplitCross) bn = kSplitCross;             // main and cross-term accumulators share one 256-column stage
  if (bn < 16 || Nout > kMaxBias) return p;
  p.n_tiles = (Nout + bn - 1) / bn;
  p.block_n = (((Nout + p.n_tiles - 1) / p.n_tiles) + 15) / 16 * 16;
  const size_t w_bytes = (size_t)2 * num_kb * p.block_n * kBlockK * 2;
  p.stages = (int)((budget - fixed - w_bytes) / (2 * kABytes));
  if (p.stages > kWsMaxStages) p.stages = kWsMaxStages;
  p.smem = fixed + w_bytes + (size_t)p.stages * 2 * kABytes;
  p.ok = p.stages >= 2 && p.n_tiles <= kNumSMs;
  return p;
}
bool linear_split_ok(int K, int Nout) { return plan_linear_split(K, Nout).ok; }

int launch_linear_split(const void* A2, int64_t lda, const float* amax_a, int M, int K, const void* W2, int64_t ldw,
                        const float* amax_w, int Nout, const float* bias, int act, float* C, int64_t ldc, cudaStream_t s) {
  const SplitPlan p = plan_linear_split(K, Nout);
  if (!p.ok) return EDG_ERR_UNSUPPORTED;
  const int k_lo = (int)(lda / 2);
  if ((lda & 127) || ldw != lda || k_lo < K) return EDG_ERR_ARG;       // hi and lo halves on 64-element boundaries
  CUtensorMap ma, mw;
  int rc = make_map_bf16(&ma, A2, M, lda, lda, kBlockK, kBlockM);     // 16-bit elements; the type only names the OOB fill
  if (rc) return rc;
  rc = make_map_bf16(&mw, W2, Nout, ldw, ldw, kBlockK, p.block_n);
  if (rc) return rc;
  if (int rc_ = ensure_dyn_smem((const void*)linear_ws_kernel<float, true>, 227 * 1024)) return rc_;
  const int m_tiles = (M + kBlockM - 1) / kBlockM;
  int groups = kNumSMs / p.n_tiles;
  if (groups > m_tiles) groups = m_tiles;
  const uint32_t idesc = make_idesc_bf16(kBlockM, p.block_n, 0, 0, /*f16=*/true);
  linear_ws_kernel<float, true><<<groups * p.n_tiles, kLinThreads, p.smem, s>>>(ma, mw, M, K, Nout, p.block_n, p.n_tiles,
                                                                                 m_tiles, p.stages, idesc, bias, act, C, ldc,
                                                                                 k_lo, amax_a, amax_w);
  return check_launch();
}

int launch_linear_tc(const void* A, int64_t lda, int M, int K, const void* W, int64_t ldw, int Nout,
                     const float* bias, int act, void* C, int c_dtype, int64_t ldc, cudaStream_t s) {
  if (Nout > kMaxBias) return EDG_ERR_UNSUPPORTED;
  int n_tiles = 1;
  const int block_n = pick_block_n(Nout, 16, &n_tiles);
  CUtensorMap ma, mw;
  int rc = make_map_bf16(&ma, A, M, K, lda, kBlockK, kBlockM);
  if (rc) return rc;
  rc = make_map_bf16(&mw, W, Nout, K, ldw, kBlockK, block_n);
  if (rc) return rc;
  // weight-stationary variant when one N tile of the weight plus >= 4 activation stages fit in shared memory
  {
    const int num_kb = (K + kBlockK - 1) / kBlockK;
    const size_t w_bytes = (size_t)num_kb * block_n * kBlockK * 2;
    const size_t fixed = 1024 + kMaxBias * sizeof(float) + 512;
    const size_t budget = 227 * 1024;
    if (w_bytes + fixed + 4 * kABytes <= budget && n_tiles <= kNumSMs && M >= 4 * kBlockM) {
      int stages = (int)((budget - fixed - w_bytes) / kABytes);
      if (stages > kWsMaxStages) stages = kWsMaxStages;
      const size_t smem = fixed + w_bytes + (size_t)stages * kABytes;
      if (c_dtype == EDG_F32) return launch_linear_ws_t<float>(ma, mw, M, K, Nout, block_n, n_tiles, stages, smem, bias, act, C, ldc, s);
      if (c_dtype == EDG_BF16) return launch_linear_ws_t<__nv_bfloat16>(ma, mw, M, K, Nout, block_n, n_tiles, stages, smem, bias, act, C, ldc, s);
      return EDG_ERR_DTYPE;
    }
  }
  if (c_dtype == EDG_F32) return launch_linear_tc_t<float>(ma, mw, M, K, Nout, block_n, n_tiles, bias, act, C, ldc, s);
  if (c_dtype == EDG_BF16) return launch_linear_tc_t<__nv_bfloat16>(ma, mw, M, K, Nout, block_n, n_tiles, bias, act, C, ldc, s);
  return EDG_ERR_DTYPE;
}

struct WgradPlan { int block_n, n_tiles, m_tiles, splits, rows_per; };
// `max_rows` > 0 caps the rows one CTA accumulates (the fp32-parity mode keeps the accumulation chains short: the
// tensor core truncates on every accumulate, so the error grows with the chain), in whole waves of the usual split
static WgradPlan plan_wgrad_tc(int R, int K1, int K2, int max_rows = 0) {
  WgradPlan p;
  p.block_n = pick_block_n(K2, 64, &p.n_tiles);
  p.m_tiles = (K1 + kBlockM - 1) / kBlockM;
  const int tiles = p.m_tiles * p.n_tiles;
  int want = (kNumSMs + tiles - 1) / tiles;
  int maxs = (R + 4 * kBlockK - 1) / (4 * kBlockK);
  p.splits = want < maxs ? want : maxs;
  if (p.splits < 1) p.splits = 1;
  p.rows_per = (((R + p.splits - 1) / p.splits) + kBlockK - 1) / kBlockK * kBlockK;
  if (max_rows > 0 && p.rows_per > max_rows) {
    const int waves = (p.rows_per + max_rows - 1) / max_rows;
    p.rows_per = (((R + p.splits * waves - 1) / (p.splits * waves)) + kBlockK - 1) / kBlockK * kBlockK;
  }
  p.splits = (R + p.rows_per - 1) / p.rows_per;
  if (p.splits < 1) p.splits = 1;
  return p;
}
// defined in edg_gemm_simt.cu
void launch_split_reduce_bias(const float* partial, int splits, int K1, int K2, int K1e, int K2e, float* dW, int64_t lddw,
                              float* dbias, int bias_of, int accumulate, cudaStream_t s);

struct TallPlan { bool ok; int m_tiles, block_n, n_tiles, splits, rows_per; };
static TallPlan plan_wgrad_tall(int R, int K1e, int K2e, int max_rows = 0) {
  TallPlan p;
  p.m_tiles = (K1e + kBlockM - 1) / kBlockM;
  p.ok = p.m_tiles <= kTallMaxM && R >= 64 * kNumSMs;          // big activations only; small ones keep wgrad_tc
  p.block_n = 160;
  while (p.block_n > 32 && (p.block_n - 32) * 1 >= K2e) p.block_n -= 32;
  if (p.m_tiles * p.block_n > kTmemCols) p.ok = false;
  p.n_tiles = (K2e + p.block_n - 1) / p.block_n;
  int want = kNumSMs / p.n_tiles;
  if (want < 1) want = 1;
  p.rows_per = (((R + want - 1) / want) + kBlockK - 1) / kBlockK * kBlockK;
  if (max_rows > 0 && p.rows_per > max_rows) {
    const int waves = (p.rows_per + max_rows - 1) / max_rows;
    p.rows_per = (((R + want * waves - 1) / (want * waves)) + kBlockK - 1) / kBlockK * kBlockK;
  }
  p.splits = (R + p.rows_per - 1) / p.rows_per;
  return p;
}

size_t wgrad_tc_workspace(int R, int K1, int K2, int max_rows) {
  size_t best = 0;
  for (int v = 0; v < 3; ++v) {
    const int K1e = K1 + (v == 2), K2e = K2 + (v == 1);
    TallPlan t = plan_wgrad_tall(R, K1e, K2e, max_rows);
    if (t.ok) {
      const size_t b = (size_t)t.splits * K1e * K2e * sizeof(float);
      if (b > best) best = b;
    }
  }                                      // the plan depends on where the ones row / column sits
  for (int v = 0; v < 3; ++v) {
    const int K1e = K1 + (v == 2), K2e = K2 + (v == 1);
    WgradPlan p = plan_wgrad_tc(R, K1e, K2e, max_rows);
    const size_t b = (size_t)p.splits * K1e * K2e * sizeof(float);
    if (b > best) best = b;
  }
  return best;
}
size_t wgrad_tc_workspace(int R, int K1, int K2) { return wgrad_tc_workspace(R, K1, K2, 0); }

// the GEMM launch alone: partial sums [slabs][K1e][K2e] into `partial`; `plant` = write the ones row / column
static int run_wgrad_tc(const void* A, int64_t lda, int K1, const void* B, int64_t ldb, int K2, int R, int bias_of,
                        bool plant, bool f16, int max_rows, float* partial, int* slabs, cudaStream_t s) {
  if (int rc_ = ensure_dyn_smem((const void*)wgrad_tc_kernel, kSmemBytes)) return rc_;
  const int K1e = K1 + (bias_of == 2 ? 1 : 0), K2e = K2 + (bias_of == 1 ? 1 : 0);
  const int ones_a = (plant && bias_of == 2) ? K1 : -1, ones_b = (plant && bias_of == 1) ? K2 : -1;
  const TallPlan t = plan_wgrad_tall(R, K1e, K2e, max_rows);
  if (t.ok) {
    if (int rc_ = ensure_dyn_smem((const void*)wgrad_tall_kernel, kTallSmem)) return rc_;
    CUtensorMap ma, mb;
    int rc = make_map_bf16(&ma, A, R, K1, lda, 64, kBlockK);
    if (rc) return rc;
    rc = make_map_bf16(&mb, B, R, K2, ldb, 32, kBlockK, /*swizzle64=*/true);
    if (rc) return rc;
    const uint32_t idesc = make_idesc_bf16(kBlockM, t.block_n, 1, 1, f16);
    wgrad_tall_kernel<<<dim3(t.n_tiles, t.splits), kThreads, kTallSmem, s>>>(ma, mb, R, K1e, K2e, t.m_tiles, t.block_n,
                                                                            t.rows_per, idesc, ones_a, ones_b, partial);
    *slabs = t.splits;
    return check_launch();
  }
  WgradPlan p = plan_wgrad_tc(R, K1e, K2e, max_rows);
  CUtensorMap ma, mb;
  int rc = make_map_bf16(&ma, A, R, K1, lda, 64, kBlockK);      // true widths: columns >= K are zero-filled
  if (rc) return rc;
  rc = make_map_bf16(&mb, B, R, K2, ldb, 64, kBlockK);
  if (rc) return rc;
  const uint32_t idesc = make_idesc_bf16(kBlockM, p.block_n, 1, 1, f16);
  dim3 grid(p.m_tiles, p.n_tiles, p.splits);
  wgrad_tc_kernel<<<grid, kThreads, kSmemBytes, s>>>(ma, mb, R, K1e, K2e, p.block_n, p.rows_per, idesc, ones_a, ones_b, partial);
  *slabs = p.splits;
  return check_launch();
}

int launch_wgrad_tc(const void* A, int64_t lda, int K1, const void* B, int64_t ldb, int K2, int R, float* dW,
                    int64_t lddw, float* dbias, int bias_of, int accumulate, float* ws, cudaStream_t s) {
  int slabs = 0;
  if (int rc = run_wgrad_tc(A, lda, K1, B, ldb, K2, R, bias_of, true, false, 0, ws, &slabs, s)) return rc;
  const int K1e = K1 + (bias_of == 2 ? 1 : 0), K2e = K2 + (bias_of == 1 ? 1 : 0);
  launch_split_reduce_bias(ws, slabs, K1, K2, K1e, K2e, dW, lddw, dbias, bias_of, accumulate, s);
  return check_launch();
}

// defined in edg_split.cu
void launch_split_reduce_bias_scaled(const float* partial, int slabs, int K1, int K2, int K1e, int K2e, float* dW,
                                     int64_t lddw, float* dbias, int bias_of, const float* amax_a, const float* amax_b,
                                     cudaStream_t s);

// split operands: a^T b = (a_hi^T b_hi + a_hi^T b_lo + a_lo^T b_hi) / (s_a s_b); three GEMM launches into
// consecutive partial-sum slabs, one scaled reduction.  The ones row / column rides on the hi and lo parts of the
// operand it sums (launches 0 and 1 for b, 0 and 2 for a), never twice on the same part.
constexpr int kSplitMainRows = 768;    // hi x hi: at most 48 accumulation steps per CTA (the cross terms are 2^-11 smaller)
size_t wgrad_split_workspace(int R, int K1, int K2) {
  return wgrad_tc_workspace(R, K1, K2, kSplitMainRows) + 2 * wgrad_tc_workspace(R, K1, K2, 0);
}

int launch_wgrad_split(const void* A2, int64_t lda, const float* amax_a, int K1, const void* B2, int64_t ldb,
                       const float* amax_b, int K2, int R, float* dW, int64_t lddw, float* dbias, int bias_of, float* ws,
                       cudaStream_t s) {
  const int ka = (int)(lda / 2), kb = (int)(ldb / 2);
  if ((lda & 127) || (ldb & 127) || ka < K1 || kb < K2) return EDG_ERR_ARG;
  const uint16_t* A = (const uint16_t*)A2;
  const uint16_t* B = (const uint16_t*)B2;
  const int K1e = K1 + (bias_of == 2 ? 1 : 0), K2e = K2 + (bias_of == 1 ? 1 : 0);
  const size_t slab = (size_t)K1e * K2e;
  int n0 = 0, n1 = 0, n2 = 0;
  // bias_of 2 = column sums of b (ones row on the a side): wanted for b_hi (launch 0) and b_lo (launch 1)
  // bias_of 1 = column sums of a (ones column on the b side): wanted for a_hi (launch 0) and a_lo (launch 2)
  if (int rc = run_wgrad_tc(A, lda, K1, B, ldb, K2, R, bias_of, true, true, kSplitMainRows, ws, &n0, s)) return rc;
  if (int rc = run_wgrad_tc(A, lda, K1, B + kb, ldb, K2, R, bias_of, bias_of == 2, true, 0, ws + (size_t)n0 * slab, &n1, s)) return rc;
  if (int rc = run_wgrad_tc(A + ka, lda, K1, B, ldb, K2, R, bias_of, bias_of == 1, true, 0, ws + (size_t)(n0 + n1) * slab, &n2, s)) return rc;
  launch_split_reduce_bias_scaled(ws, n0 + n1 + n2, K1, K2, K1e, K2e, dW, lddw, dbias, bias_of, amax_a, amax_b, s);
  return check_launch();
}

// defined in edg_gemm_simt.cu
void launch_split_reduce_bias_batch(const float* partial, int n, int splits, int K1, int K2, int K1e, int K2e,
                                    float* const* dW, int64_t lddw, float* const* dbias, int bias_of, cudaStream_t s);

size_t wgrad_tc_batch_workspace(int n, int R, int K1, int K2) {
  size_t best = 0;
  for (int v = 0; v < 3; ++v) {
    const int K1e = K1 + (v == 2), K2e = K2 + (v == 1);
    WgradPlan p = plan_wgrad_tc(R, K1e, K2e);
    const size_t b = (size_t)p.splits * K1e * K2e * sizeof(float);
    if (b > best) best = b;
  }
  return best * (size_t)n;
}

int launch_wgrad_tc_batch(int n, const void* const* A, int64_t lda, int K1, const void* const* B, int64_t ldb, int K2, int R,
                          float* const* dW, int64_t lddw, float* const* dbias, int bias_of, float* ws, cudaStream_t s) {
  if (n > kWgradBatchMax) return EDG_ERR_UNSUPPORTED;
  if (int rc_ = ensure_dyn_smem((const void*)wgrad_tc_batch_kernel, kSmemBytes)) return rc_;
  const int K1e = K1 + (bias_of == 2 ? 1 : 0), K2e = K2 + (bias_of == 1 ? 1 : 0);
  WgradPlan p = plan_wgrad_tc(R, K1e, K2e);
  // the problems share the SMs: fewer row splits per problem keep the partial-sum traffic down
  int splits = (kNumSMs + p.m_tiles * p.n_tiles * n - 1) / (p.m_tiles * p.n_tiles * n);
  if (splits > p.splits) splits = p.splits;
  if (splits < 1) splits = 1;
  const int rows_per = (((R + splits - 1) / splits) + kBlockK - 1) / kBlockK * kBlockK;
  splits = (R + rows_per - 1) / rows_per;
  WgradBatchMaps maps;
  memset(&maps, 0, sizeof(maps));
  for (int i = 0; i < n; ++i) {
    int rc = make_map_bf16(&maps.a[i], A[i], R, K1, lda, 64, kBlockK);
    if (rc) return rc;
    rc = make_map_bf16(&maps.b[i], B[i], R, K2, ldb, 64, kBlockK);
    if (rc) return rc;
  }
  const uint32_t idesc = make_idesc_bf16(kBlockM, p.block_n, 1, 1);
  dim3 grid(p.m_tiles, p.n_tiles, splits * n);
  wgrad_tc_batch_kernel<<<grid, kThreads, kSmemBytes, s>>>(maps, splits, R, K1e, K2e, p.block_n, rows_per, idesc,
                                                           bias_of == 2 ? K1 : -1, bias_of == 1 ? K2 : -1, ws);
  launch_split_reduce_bias_batch(ws, n, splits, K1, K2, K1e, K2e, dW, lddw, dbias, bias_of, s);
  return check_launch();
}

}  // namespace edg
