// Sentence-window staging shared by the row-streaming kernels of the gated block.
//
// A block owns the sentences that START inside a window of `tile_rows` packed rows.  Their rows are
// contiguous in memory, so ONE bulk asynchronous copy (cp.async.bulk on the TMA engine, mbarrier
// completion) brings them into shared memory; all per-row work then runs on 128-bit shared-memory
// loads.  DRAM latency is paid once per window and hidden by the other resident blocks, instead of
// once per row of a sequential per-sentence loop.
//
// Every sentence has exactly one owner, empty ones (0 rows) included: window 0 also owns the empty sentences
// before the first row, and a window that lies inside one long sentence owns the empty sentences that start at its
// end.  Such a window has no rows to stage (r1 <= r0) and issues no copy, but it still writes the outputs of its
// sentences (all of them empty); it must then not wait on the barrier (has_rows() is false).
#pragma once
#include "edg_common.cuh"

namespace edg {

struct RowWindow {
  int r0, r1, s0, s1;
  __device__ __forceinline__ bool has_rows() const { return r1 > r0; }   // false: no copy was issued, do not wait
};

__device__ __forceinline__ uint32_t stg_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// Called by every thread of the block.  `sh` = 4 ints and `bar` = one mbarrier in static shared memory.
// The host guarantees cap_rows >= tile_rows + max_len - 1, so the window always fits.
template <typename T>
__device__ __forceinline__ RowWindow stage_window(const T* __restrict__ x, int64_t ldx, int N, int B, int tile_rows,
                                                  const int32_t* __restrict__ sent_ptr, const int32_t* __restrict__ row_sent,
                                                  uint8_t* smem_rows, uint64_t* bar, int* sh) {
  if (threadIdx.x == 0 && threadIdx.y == 0) {
    const int w0 = blockIdx.x * tile_rows, w1 = w0 + tile_rows;
    // first sentence starting at or after w0 / w1.  Two levels of dependent loads only (the copy cannot start before
    // them): both row_sent lookups together, then sent_ptr[s] and sent_ptr[s + 1] of both speculatively.
    const int a0 = w0 < N ? __ldg(row_sent + w0) : B, a1 = w1 < N ? __ldg(row_sent + w1) : B;
    const int p0 = __ldg(sent_ptr + a0), q0 = a0 < B ? __ldg(sent_ptr + a0 + 1) : p0;
    const int p1 = __ldg(sent_ptr + a1), q1 = a1 < B ? __ldg(sent_ptr + a1 + 1) : p1;
    const bool up0 = w0 < N && p0 < w0, up1 = w1 < N && p1 < w1;
    const int s0 = w0 == 0 ? 0 : a0 + up0, s1 = a1 + up1;     // row_sent names no leading empty sentence
    const int r0 = up0 ? q0 : p0, r1 = up1 ? q1 : p1;
    sh[0] = r0; sh[1] = r1; sh[2] = s0; sh[3] = s1;
    const uint32_t b32 = stg_smem_u32(bar);
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(b32));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    if (r1 > r0) {
      const uint32_t bytes = (uint32_t)(r1 - r0) * (uint32_t)(ldx * sizeof(T));
      asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(b32), "r"(bytes) : "memory");
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                   ::"r"(stg_smem_u32(smem_rows)), "l"(x + (int64_t)r0 * ldx), "r"(bytes), "r"(b32) : "memory");
    }
  }
  __syncthreads();
  RowWindow w;
  w.r0 = sh[0]; w.r1 = sh[1]; w.s0 = sh[2]; w.s1 = sh[3];
  return w;
}

__device__ __forceinline__ void wait_window(uint64_t* bar) {
  const uint32_t b32 = stg_smem_u32(bar);
  uint32_t ok = 0;
  while (!ok) {
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(ok) : "r"(b32) : "memory");
  }
}

// 16 bytes of the activation dtype from shared memory -> fp32 lanes
template <typename T> struct SVec16;
template <> struct SVec16<float> {
  __device__ static __forceinline__ void load(uint32_t saddr, float (&f)[4]) {
    uint32_t a, b, c, d;
    asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(a), "=r"(b), "=r"(c), "=r"(d) : "r"(saddr));
    f[0] = __uint_as_float(a); f[1] = __uint_as_float(b); f[2] = __uint_as_float(c); f[3] = __uint_as_float(d);
  }
};
template <> struct SVec16<__nv_bfloat16> {
  __device__ static __forceinline__ void load(uint32_t saddr, float (&f)[8]) {
    uint32_t w[4];
    asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(w[0]), "=r"(w[1]), "=r"(w[2]), "=r"(w[3]) : "r"(saddr));
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      f[2 * i] = __uint_as_float(w[i] << 16);
      f[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
    }
  }
};

// (A persistent one-block-per-SM variant with a 3-stage ring of windows was measured and rejected: 56-74 us vs
// 42-44 us for aggregation at C2 -- with ~70-row windows the block-wide barriers outweigh the hidden prologue.)
// host side: window geometry for a row pitch (bytes) and the longest sentence; tile_rows < 8 = do not stage
struct WindowPlan { int tile_rows, cap_rows; size_t smem_rows; };
inline WindowPlan plan_window(size_t pitch_bytes, int max_len, size_t extra_per_row = 0, size_t fixed_extra = 0) {
  WindowPlan p;
  // ~72 KB per block keeps 3 blocks per SM resident; long sentences get one ~200 KB block per SM
  p.cap_rows = (72 * 1024 > fixed_extra) ? (int)((72 * 1024 - fixed_extra) / (pitch_bytes + extra_per_row)) : 0;
  p.tile_rows = p.cap_rows - max_len + 1;
  if (p.tile_rows < 16) {
    p.cap_rows = (200 * 1024 > fixed_extra) ? (int)((200 * 1024 - fixed_extra) / (pitch_bytes + extra_per_row)) : 0;
    p.tile_rows = p.cap_rows - max_len + 1;
  }
  p.smem_rows = (size_t)p.cap_rows * pitch_bytes;
  return p;
}

}  // namespace edg
