// Shared device/host helpers for libedgcn (sm_100a only).
#pragma once

#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/edgcn.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "libedgcn is written for sm_100a only"
#endif

namespace edg {

constexpr int kNumSMs = 148;   // B200: 2 dies x 74 SMs

// ---- host side ------------------------------------------------------------
void set_cuda_error(cudaError_t e);

inline int check_launch() {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    set_cuda_error(e);
    return EDG_ERR_CUDA;
  }
  return EDG_OK;
}

// Opt a kernel into `smem` bytes of dynamic shared memory (> 48 KB needs cudaFuncSetAttribute).  The attribute is per
// (device, function): the cache is keyed by both, so a second GPU in the same process gets its own opt-in; thread-safe
// (autograd calls backward from another host thread).
int ensure_dyn_smem(const void* kernel, size_t smem);

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }
inline size_t dtype_size(int dt) { return dt == EDG_BF16 ? 2 : 4; }
inline bool row_pitch_ok(int dt, int64_t ld) { return (ld * (int64_t)dtype_size(dt)) % 16 == 0; }
inline int64_t ceil_div64(int64_t a, int64_t b) { return (a + b - 1) / b; }

// ---- device side ------------------------------------------------------------
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// 16-byte vector of the activation dtype <-> fp32 lanes
template <typename T> struct Vec16;
template <> struct Vec16<float> {
  static constexpr int kElems = 4;
  __device__ static __forceinline__ void load(const float* p, float (&f)[4]) {
    float4 v = __ldg(reinterpret_cast<const float4*>(p));
    f[0] = v.x; f[1] = v.y; f[2] = v.z; f[3] = v.w;
  }
  __device__ static __forceinline__ void store(float* p, const float (&f)[4]) {
    *reinterpret_cast<float4*>(p) = make_float4(f[0], f[1], f[2], f[3]);
  }
};
template <> struct Vec16<__nv_bfloat16> {
  static constexpr int kElems = 8;
  __device__ static __forceinline__ void load(const __nv_bfloat16* p, float (&f)[8]) {
    uint4 v = __ldg(reinterpret_cast<const uint4*>(p));
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {   // bf16 -> fp32 is a 16-bit shift
      f[2 * i] = __uint_as_float(w[i] << 16);
      f[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
    }
  }
  __device__ static __forceinline__ void store(__nv_bfloat16* p, const float (&f)[8]) {
    uint32_t w[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      __nv_bfloat162 h = __floats2bfloat162_rn(f[2 * i], f[2 * i + 1]);
      w[i] = *reinterpret_cast<uint32_t*>(&h);
    }
    *reinterpret_cast<uint4*>(p) = make_uint4(w[0], w[1], w[2], w[3]);
  }
};

// lo += bf16(low half of w), hi += bf16(high half): the mixed-precision add of sm_100 (`add.f32.bf16`, SASS FHADD.BF16
// with a half-register operand) -- one instruction per element where shift/mask + FADD needs two, bit-identical result
// (bf16 -> fp32 is exact).  The row-summing loops of this library are issue-slot bound on exactly that unpack.
__device__ __forceinline__ void add_bf16x2(uint32_t w, float& lo, float& hi) {
  asm("{\n\t.reg .b16 l, h;\n\tmov.b32 {l, h}, %2;\n\tadd.rn.f32.bf16 %0, l, %0;\n\tadd.rn.f32.bf16 %1, h, %1;\n\t}"
      : "+f"(lo), "+f"(hi) : "r"(w));
}

__device__ __forceinline__ float to_f32(float v) { return v; }
__device__ __forceinline__ float to_f32(__nv_bfloat16 v) { return __bfloat162float(v); }
template <typename T> __device__ __forceinline__ T from_f32(float v);
template <> __device__ __forceinline__ float from_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ __nv_bfloat16 from_f32<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }

// runtime-dtype scalar access (small [B,D]-sized helpers only)
__device__ __forceinline__ float load_as_f32(const void* p, int dtype, int64_t idx) {
  return dtype == EDG_BF16 ? __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(p)[idx])
                           : reinterpret_cast<const float*>(p)[idx];
}
__device__ __forceinline__ void store_from_f32(void* p, int dtype, int64_t idx, float v) {
  if (dtype == EDG_BF16) reinterpret_cast<__nv_bfloat16*>(p)[idx] = __float2bfloat16_rn(v);
  else reinterpret_cast<float*>(p)[idx] = v;
}

__device__ __forceinline__ float sigmoidf_(float x) { return 1.0f / (1.0f + expf(-x)); }

// ---- gate dropout mask (include/edgcn.h, edg_dropout_rows) ----------------------------------------------------
// keep(seed, stream, row, column) is a counter-based hash, so every kernel that applies or differentiates the mask
// regenerates it where it needs it and nothing is stored.  The format is restated bit for bit by the tests (numpy).
__host__ __device__ __forceinline__ uint32_t mix32(uint32_t x) {
  x ^= x >> 16; x *= 0x7feb352dU; x ^= x >> 15; x *= 0x846ca68bU; x ^= x >> 16;
  return x;
}
struct DropKey { uint32_t lo, hi; };
// the per-stream key from the DEVICE seed (a captured graph reads a new seed on every replay)
__device__ __forceinline__ DropKey dropout_key(const int64_t* seed, uint32_t stream_id) {
  const uint64_t sd = (uint64_t)__ldg(seed);
  return DropKey{(uint32_t)sd ^ (stream_id * 0xC2B2AE3DU), (uint32_t)(sd >> 32)};
}
__device__ __forceinline__ bool dropout_keep(DropKey k, uint32_t row, uint32_t col, uint32_t thr) {
  const uint32_t u = mix32(mix32(row * 0x9E3779B1U + k.lo) ^ (col * 0x85EBCA77U + k.hi));
  return u >= thr;
}
// an element is kept when its hash is >= floor(p * 2^32); p in [0, 1)
inline uint32_t dropout_threshold(float p) {
  const double t = (double)p * 4294967296.0;
  return t >= 4294967295.0 ? 4294967295U : (uint32_t)t;
}
inline bool dropout_p_ok(float p) { return p >= 0.f && p < 1.f; }

}  // namespace edg
