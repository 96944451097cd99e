// Sentence-window (shared-memory staged) versions of the row-streaming kernels of the gated block:
// gated max-pool views, importance scores + softmax product, and the head backward.  Same arithmetic as
// the per-sentence kernels in edg_block.cu (which remain for sentences too long for a window); the rows
// come from ONE bulk async copy per window instead of a dependent global load per row.
#include <math.h>

#include "edg_staged.cuh"

namespace edg {

template <int I64> __device__ __forceinline__ float sdist_at(const void* dist, int64_t i) {
  return I64 ? (float)__ldg(reinterpret_cast<const long long*>(dist) + i) : (float)__ldg(reinterpret_cast<const int32_t*>(dist) + i);
}

// ---- gated max-pool views (bert_amir5.py:627-636, :640) -------------------------------------------
// thread = (16-byte column chunk x, sentence lane y).  Gates are sigmoid outputs (> 0) and rounding is monotone,
// so max_t fl(h_t * g) = fl((max_t h_t) * g): ONE gate-independent pass finds the column maximum m and its first
// row; every view is then a single multiply (3 instructions per element per row instead of 4 per view).  The
// arg-max row equals torch.max's unless two DIFFERENT values of h round to the same product, where either row is
// an exact maximiser; a gate that underflowed to 0 makes every product 0 and the first row wins, as in torch.
template <typename T, int V>
__global__ void __launch_bounds__(256)
pool_staged_kernel(const T* __restrict__ h, int64_t ldh, const int32_t* __restrict__ sent_ptr,
                   const int32_t* __restrict__ row_sent, int N, int B, int D, int tile_rows, int cap_rows,
                   const float* __restrict__ gates, float* __restrict__ pooled, int32_t* __restrict__ arg,
                   float* __restrict__ hmax) {
  constexpr int E = Vec16<T>::kElems;
  extern __shared__ __align__(128) uint8_t win[];
  __shared__ __align__(8) uint64_t bar;
  __shared__ int sh[4];
  const RowWindow w = stage_window<T>(h, ldh, N, B, tile_rows, sent_ptr, row_sent, win, &bar, sh);
  const int pitch = (int)(ldh * (int64_t)sizeof(T));
  const int c = threadIdx.x * E;
  const int64_t BD = (int64_t)B * D;
  const uint32_t xs = stg_smem_u32(win) + threadIdx.x * 16;
  bool waited = !w.has_rows();           // a window without rows still writes its (empty) sentences
  for (int s = w.s0 + threadIdx.y; s < w.s1; s += blockDim.y) {
    const int beg = __ldg(sent_ptr + s), end = __ldg(sent_ptr + s + 1);
    // the gate vectors do not depend on the window: issue their loads BEFORE blocking on the bulk copy
    float g[V][E];
#pragma unroll
    for (int v = 0; v < V; ++v)
#pragma unroll
      for (int k = 0; k < E; ++k) g[v][k] = (c + k < D) ? __ldg(gates + v * BD + (int64_t)s * D + c + k) : 0.f;
    if (!waited) { wait_window(&bar); waited = true; }
    float m[E];
    int32_t where[E];
#pragma unroll
    for (int k = 0; k < E; ++k) { m[k] = -INFINITY; where[k] = beg; }
    uint32_t addr = xs + (uint32_t)((beg - w.r0) * pitch);
    for (int t = beg; t < end; ++t, addr += pitch) {
      float f[E];
      SVec16<T>::load(addr, f);
#pragma unroll
      for (int k = 0; k < E; ++k)
        if (f[k] > m[k]) { m[k] = f[k]; where[k] = t; }                  // strict: first row wins ties
    }
#pragma unroll
    for (int v = 0; v < V; ++v)
#pragma unroll
      for (int k = 0; k < E; ++k)
        if (c + k < D) {
          const int64_t o = v * BD + (int64_t)s * D + c + k;
          pooled[o] = (beg < end) ? m[k] * g[v][k] : 0.f;
          arg[o] = (beg < end) ? (g[v][k] != 0.f ? where[k] : beg) : -1;
        }
    if (hmax)
#pragma unroll
      for (int k = 0; k < E; ++k)
        if (c + k < D) hmax[(int64_t)s * D + c + k] = (beg < end) ? m[k] : 0.f;
  }
  if (!waited) wait_window(&bar);        // never leave a bulk copy in flight into a dead block
}

// ---- importance scores, softmax product, and d kl / d (v, c) units (bert_amir5.py:645-648) ----------
// One WARP per sentence of the window, no block barrier after the window has landed:
//   P1 scores: LANE = ROW.  Every lane walks its own row's 16-byte chunks (the sentence's weights gate*v are broadcast
//      reads of a per-warp shared-memory copy), so a row's dot product needs no shuffle reduction and the scores end up
//      one per lane -- the layout the softmax wants.  Four accumulators keep the FMA chain short.
//   P2 softmax statistics over the lanes: kl_b and u_t = P_t (Q_t - kl_b) / B.
//   P3 sf = sum_t u_t h_t: lanes = chunks, u_t broadcast by shuffle from the lane that owns row t.
// (The first version -- window-wide phases, warp per ROW in P1, three block barriers -- spent 32 % of its samples in
// barriers and needed 25.5 M warp instructions per launch at config 2; this one needs ~8 M.)
constexpr int kSMaxQ = 4;                  // 16-byte chunks per lane in P3 (chunks <= 128)
constexpr int kSMaxPass = 4;               // rows per sentence <= 128 (lane = row, four passes)
constexpr int kScoresWarps = 4;            // warps per block: a 72 KB window holds ~2.6 sentences of config 2

template <typename T, int I64, int Q>
__global__ void __launch_bounds__(32 * kScoresWarps)
scores_staged_kernel(const T* __restrict__ h, int64_t ldh, const int32_t* __restrict__ sent_ptr,
                     const int32_t* __restrict__ row_sent, int N, int B, int D, int chunks, int tile_rows, int cap_rows,
                     const float* __restrict__ gate, const float* __restrict__ vvec, const float* __restrict__ cvec,
                     const void* __restrict__ dist, float* __restrict__ scores, float* __restrict__ kl_b,
                     float* __restrict__ dv_unit, float* __restrict__ dc_unit, float* __restrict__ u_unit,
                     float* __restrict__ sf_unit) {
  constexpr int E = Vec16<T>::kElems;
  extern __shared__ __align__(128) uint8_t win[];
  __shared__ __align__(8) uint64_t bar;
  __shared__ int sh[4];
  const RowWindow w = stage_window<T>(h, ldh, N, B, tile_rows, sent_ptr, row_sent, win, &bar, sh);
  const int pitch = (int)(ldh * (int64_t)sizeof(T));
  const int lane = threadIdx.x, warp = threadIdx.y;
  const int width = chunks * E;
  float* w_s = reinterpret_cast<float*>(win + (size_t)cap_rows * pitch) + (size_t)warp * width;   // this warp's gate*v
  const uint32_t w_a = stg_smem_u32(w_s);
  const uint32_t xs = stg_smem_u32(win);
  const float invB = 1.0f / (float)B;
  bool waited = !w.has_rows();           // a window without rows still writes its (empty) sentences
  for (int s = w.s0 + warp; s < w.s1; s += kScoresWarps) {
    const int beg = __ldg(sent_ptr + s) - w.r0, end = __ldg(sent_ptr + s + 1) - w.r0;
    const int n = end - beg;
    // the sentence's weights and distances do not depend on the window: their loads are issued before the bulk-copy wait
    __syncwarp();
    float gq[Q][E];                                       // this lane's gate entries (chunks lane, lane + 32, ...)
    {
      float vq[Q][E];
#pragma unroll
      for (int q = 0; q < Q; ++q)                         // all loads first: ONE global round trip per sentence
#pragma unroll
        for (int k = 0; k < E; ++k) {
          const int i = (lane + 32 * q) * E + k;
          const bool ok = lane + 32 * q < chunks && i < D;
          gq[q][k] = ok ? __ldg(gate + (int64_t)s * D + i) : 0.f;
          vq[q][k] = ok ? __ldg(vvec + (int64_t)s * D + i) : 0.f;
        }
#pragma unroll
      for (int q = 0; q < Q; ++q)
        if (lane + 32 * q < chunks) {
#pragma unroll
          for (int k = 0; k < E; ++k) w_s[(lane + 32 * q) * E + k] = gq[q][k] * vq[q][k];
        }
    }
    const float cb = cvec ? __ldg(cvec + s) : 0.f;
    float dq[kSMaxPass];
#pragma unroll
    for (int p = 0; p < kSMaxPass; ++p) dq[p] = (32 * p + lane < n) ? sdist_at<I64>(dist, w.r0 + beg + 32 * p + lane) : -INFINITY;
    __syncwarp();
    if (!waited) { wait_window(&bar); waited = true; }
    // ---- P1
    float sc[kSMaxPass];
#pragma unroll
    for (int p = 0; p < kSMaxPass; ++p) {
      sc[p] = -INFINITY;
      if (32 * p < n) {                                   // warp-uniform
        const int t = 32 * p + lane;
        if (t < n) {
          const uint32_t ra = xs + (uint32_t)((beg + t) * pitch);
          float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll 4
          for (int c = 0; c < chunks; ++c) {
            float f[E], g[E];
            SVec16<T>::load(ra + (uint32_t)c * 16u, f);
#pragma unroll
            for (int k = 0; k < E; k += 4) SVec16<float>::load(w_a + (uint32_t)(c * E + k) * 4u, *reinterpret_cast<float(*)[4]>(&g[k]));
#pragma unroll
            for (int k = 0; k < E; k += 4) {
              a0 = fmaf(f[k], g[k], a0); a1 = fmaf(f[k + 1], g[k + 1], a1);
              a2 = fmaf(f[k + 2], g[k + 2], a2); a3 = fmaf(f[k + 3], g[k + 3], a3);
            }
          }
          const float v = ((a0 + a1) + (a2 + a3)) + cb;
          sc[p] = v;
          scores[w.r0 + beg + t] = v;
        }
      }
    }
    // ---- P2
    float ms = -INFINITY, mq = -INFINITY;
#pragma unroll
    for (int p = 0; p < kSMaxPass; ++p) { ms = fmaxf(ms, sc[p]); mq = fmaxf(mq, dq[p]); }
    ms = warp_max(ms); mq = warp_max(mq);
    float es[kSMaxPass], eq[kSMaxPass], zs = 0.f, zq = 0.f;
#pragma unroll
    for (int p = 0; p < kSMaxPass; ++p) {
      const bool ok = 32 * p + lane < n;
      es[p] = ok ? expf(sc[p] - ms) : 0.f;
      eq[p] = ok ? expf(dq[p] - mq) : 0.f;
      zs += es[p]; zq += eq[p];
    }
    zs = warp_sum(zs); zq = warp_sum(zq);
    float kacc = 0.f;
#pragma unroll
    for (int p = 0; p < kSMaxPass; ++p) kacc += (es[p] / zs) * (eq[p] / zq);
    const float klb = n > 0 ? warp_sum(kacc) : 0.f;
    if (lane == 0) kl_b[s] = klb;
    if (dv_unit == nullptr) continue;
    float u[kSMaxPass], dcu = 0.f;
#pragma unroll
    for (int p = 0; p < kSMaxPass; ++p) {
      const bool ok = 32 * p + lane < n;
      u[p] = ok ? (es[p] / zs) * ((eq[p] / zq) - klb) * invB : 0.f;
      if (ok && u_unit) u_unit[w.r0 + beg + 32 * p + lane] = u[p];
      dcu += u[p];
    }
    dcu = warp_sum(dcu);
    if (lane == 0 && dc_unit) dc_unit[s] = dcu;
    // ---- P3
    float dvu[Q][E];
#pragma unroll
    for (int q = 0; q < Q; ++q)
#pragma unroll
      for (int k = 0; k < E; ++k) dvu[q][k] = 0.f;
#pragma unroll
    for (int p = 0; p < kSMaxPass; ++p) {
      if (32 * p < n) {
        const int cnt = min(32, n - 32 * p);
        const uint32_t ra = xs + (uint32_t)((beg + 32 * p) * pitch) + (uint32_t)lane * 16u;
        // four rows per step: their shuffles and shared-memory loads are independent (one warp per sentence has no
        // other warp of the same sentence to hide a dependent chain)
#pragma unroll 1
        for (int t0 = 0; t0 < cnt; t0 += 4) {
          float ut[4];
#pragma unroll
          for (int r = 0; r < 4; ++r) ut[r] = __shfl_sync(0xffffffffu, u[p], (t0 + r) & 31);
#pragma unroll
          for (int q = 0; q < Q; ++q) {
            if (lane + 32 * q < chunks) {
              float f[4][E];
#pragma unroll
              for (int r = 0; r < 4; ++r)
                if (t0 + r < cnt) SVec16<T>::load(ra + (uint32_t)((t0 + r) * pitch) + (uint32_t)q * 512u, f[r]);
#pragma unroll
              for (int r = 0; r < 4; ++r)
                if (t0 + r < cnt) {
#pragma unroll
                  for (int k = 0; k < E; ++k) dvu[q][k] = fmaf(ut[r], f[r][k], dvu[q][k]);
                }
            }
          }
        }
      }
    }
#pragma unroll
    for (int q = 0; q < Q; ++q) {
      const int c = (lane + 32 * q) * E;
      if (lane + 32 * q < chunks) {
#pragma unroll
        for (int k = 0; k < E; ++k)
          if (c + k < D) {
            dv_unit[(int64_t)s * D + c + k] = dvu[q][k] * gq[q][k];
            if (sf_unit) sf_unit[(int64_t)s * D + c + k] = dvu[q][k];
          }
      }
    }
  }
  if (!waited) wait_window(&bar);        // never leave a bulk copy in flight into a dead block
}

// ---- head backward (scores/kl, final max-pool, optional direct x_out gradient) -----------------------
// three ~72 KB windows fit an SM; without the cap the bf16 instantiation takes 106 registers and only two blocks
// are resident (65.5 vs 70.5 us at C2 with the cap; 60 bytes of spills)
#ifndef EDG_HEAD_MINBLOCKS
#define EDG_HEAD_MINBLOCKS 3
#endif
template <typename T, int I64>
__global__ void __launch_bounds__(256, EDG_HEAD_MINBLOCKS)
head_bwd_staged_kernel(const T* __restrict__ h, int64_t ldh, const int32_t* __restrict__ sent_ptr,
                       const int32_t* __restrict__ row_sent, int N, int B, int D, int tile_rows, int cap_rows,
                       const float* __restrict__ gate, const float* __restrict__ vvec, const void* __restrict__ dist,
                       const float* __restrict__ scores, const float* __restrict__ kl_b, const float* __restrict__ g_kl,
                       const float* __restrict__ g_scores, const float* __restrict__ g_pooled, const int32_t* __restrict__ arg,
                       const T* __restrict__ g_xout, int64_t ldgx, T* __restrict__ dh, int64_t lddh,
                       float* __restrict__ dgate, float* __restrict__ dv, float* __restrict__ dc) {
  constexpr int E = Vec16<T>::kElems;
  extern __shared__ __align__(128) uint8_t win[];
  __shared__ __align__(8) uint64_t bar;
  __shared__ int sh[4];
  const RowWindow w = stage_window<T>(h, ldh, N, B, tile_rows, sent_ptr, row_sent, win, &bar, sh);
  const int pitch = (int)(ldh * (int64_t)sizeof(T));
  float* ds_s = reinterpret_cast<float*>(win + (size_t)cap_rows * pitch);      // [cap_rows] d loss / d scores
  const int nthreads = blockDim.x * blockDim.y;
  const int tid = threadIdx.y * blockDim.x + threadIdx.x;
  // only FULL warps take part in phase 1 (its reductions use full-mask shuffles); the block's last, partial
  // warp skips it.  The host launches this kernel only when the block holds at least one full warp.
  const int lane = tid & 31, wid = tid >> 5, nwarps = nthreads >> 5;
  const bool have_s = (scores != nullptr) && (g_kl != nullptr || g_scores != nullptr);
  // phase 1 (overlaps the bulk copy): ds for every row of the window, one warp per sentence
  for (int s = w.s0 + wid; wid < nwarps && s < w.s1; s += nwarps) {
    const int beg = __ldg(sent_ptr + s), end = __ldg(sent_ptr + s + 1);
    float tot = 0.f;
    if (have_s) {
      float ms = 0.f, zs = 1.f, mq = 0.f, zq = 1.f, klb = 0.f, gk = 0.f;
      if (g_kl) {
        gk = __ldg(g_kl) / (float)B;
        klb = __ldg(kl_b + s);
        ms = -INFINITY; mq = -INFINITY;
        for (int t = beg + lane; t < end; t += 32) { ms = fmaxf(ms, __ldg(scores + t)); mq = fmaxf(mq, sdist_at<I64>(dist, t)); }
        ms = warp_max(ms); mq = warp_max(mq);
        zs = 0.f; zq = 0.f;
        for (int t = beg + lane; t < end; t += 32) { zs += expf(__ldg(scores + t) - ms); zq += expf(sdist_at<I64>(dist, t) - mq); }
        zs = warp_sum(zs); zq = warp_sum(zq);
      }
      for (int t = beg + lane; t < end; t += 32) {
        float v = 0.f;
        if (g_kl) v = gk * (expf(__ldg(scores + t) - ms) / zs) * ((expf(sdist_at<I64>(dist, t) - mq) / zq) - klb);
        if (g_scores) v += __ldg(g_scores + t);
        ds_s[t - w.r0] = v;
        tot += v;
      }
      tot = warp_sum(tot);
    } else {
      for (int t = beg + lane; t < end; t += 32) ds_s[t - w.r0] = 0.f;
    }
    if (lane == 0 && dc) dc[s] = tot;
  }
  // (the block barrier that publishes ds_s and the wait on the window sit inside phase 2, after its prefetches)
  // phase 2: thread = (16-byte column chunk x, sentence lane y).  With sf = sum_t ds_t h_t (per column):
  //   dh_t = ds_t * (g v)  [+ g gp on the arg-max row]      dv = g * sf      dgate = v * sf + gp * h_arg
  // Every per-sentence vector is loaded before blocking on the window; h_arg comes from shared memory.
  const int c = threadIdx.x * E;
  const uint32_t xs = stg_smem_u32(win) + threadIdx.x * 16;
  float g[E], vv[E], gp[E];
  int32_t where[E];
  int beg = 0, end = 0;
  auto load_sentence = [&](int s) {
    beg = __ldg(sent_ptr + s); end = __ldg(sent_ptr + s + 1);
#pragma unroll
    for (int k = 0; k < E; ++k) {
      const bool ok = c + k < D;
      const int64_t o = (int64_t)s * D + c + k;
      g[k] = ok ? __ldg(gate + o) : 0.f;
      vv[k] = (ok && vvec) ? __ldg(vvec + o) : 0.f;
      gp[k] = (ok && g_pooled) ? __ldg(g_pooled + o) : 0.f;
      where[k] = (ok && g_pooled) ? __ldg(arg + o) : -1;
    }
  };
  int s = w.s0 + threadIdx.y;
  if (s < w.s1) load_sentence(s);          // in flight while the block waits below
  __syncthreads();                         // publishes ds_s (phase 1)
  if (w.has_rows()) wait_window(&bar);     // a window without rows still writes its (empty) sentences
  for (bool first = true; s < w.s1; s += blockDim.y, first = false) {
    if (!first) load_sentence(s);
    float gv[E], ggp[E], sf[E], xg[E];
#pragma unroll
    for (int k = 0; k < E; ++k) { gv[k] = g[k] * vv[k]; ggp[k] = g[k] * gp[k]; sf[k] = 0.f; xg[k] = 0.f; }
    uint32_t addr = xs + (uint32_t)((beg - w.r0) * pitch);
    for (int t = beg; t < end; ++t, addr += pitch) {
      float f[E], o[E];
      SVec16<T>::load(addr, f);
      const float dst = ds_s[t - w.r0];
      if (g_xout) {                                  // optional direct gradient on x_out = g * h
        float gx[E];
        Vec16<T>::load(g_xout + (int64_t)t * ldgx + c, gx);
#pragma unroll
        for (int k = 0; k < E; ++k) { o[k] = fmaf(dst, gv[k], g[k] * gx[k]); xg[k] = fmaf(f[k], gx[k], xg[k]); }
      } else {
#pragma unroll
        for (int k = 0; k < E; ++k) o[k] = dst * gv[k];
      }
#pragma unroll
      for (int k = 0; k < E; ++k) {
        sf[k] = fmaf(dst, f[k], sf[k]);
        if (where[k] == t) o[k] += ggp[k];           // the arg-max row also receives the pooled gradient
      }
      if (dh) Vec16<T>::store(dh + (int64_t)t * lddh + c, o);
    }
#pragma unroll
    for (int k = 0; k < E; ++k)
      if (c + k < D) {
        const int64_t o = (int64_t)s * D + c + k;
        float dg = fmaf(vv[k], sf[k], xg[k]);
        if (where[k] >= beg && where[k] < end) {      // as the per-sentence kernel: only a row of the sentence
          const T* hp = reinterpret_cast<const T*>(win + (size_t)(where[k] - w.r0) * pitch) + c + k;
          dg = fmaf(gp[k], to_f32(*hp), dg);
        }
        if (dgate) dgate[o] = dg;
        if (dv) dv[o] = g[k] * sf[k];
      }
  }
}

// ---- host launchers (called from the C-ABI functions in edg_block.cu) --------------------------------
template <typename K> static int opt_in_smem(K kernel, size_t smem, size_t*) { return ensure_dyn_smem((const void*)kernel, smem); }

static inline dim3 chunk_block(int chunks) {
  int y = 256 / chunks;
  if (y > 8) y = 8;
  if (y < 1) y = 1;
  return dim3(chunks, y);
}

// returns 1 when the staged path does not apply (caller falls back to the per-sentence kernels); N == 0 (every
// sentence empty) is one such case: it would be a grid of 0 blocks
template <typename T>
int pool_fwd_staged(const void* h, int64_t ldh, const int32_t* sent_ptr, const int32_t* row_sent, int N, int B, int D,
                    int max_len, const float* gates, int V, float* pooled, int32_t* arg, float* hmax, cudaStream_t s) {
  constexpr int E = Vec16<T>::kElems;
  const int chunks = (D + E - 1) / E;
  if (!row_sent || max_len <= 0 || N <= 0 || chunks > 256) return 1;
  const dim3 blk = chunk_block(chunks);
  const WindowPlan p = plan_window((size_t)ldh * sizeof(T), max_len);
  if (p.tile_rows < 8) return 1;
  const unsigned blocks = (unsigned)((N + p.tile_rows - 1) / p.tile_rows);
  const int64_t BD = (int64_t)B * D;
  static size_t seen[4] = {0, 0, 0, 0};
  for (int v0 = 0; v0 < V; v0 += 2) {
    const int nv = (V - v0) < 2 ? (V - v0) : 2;
    const size_t smem = p.smem_rows;
    const float* g = gates + v0 * BD;
    float* pp = pooled + v0 * BD;
    int32_t* aa = arg + v0 * BD;
    int rc = EDG_OK;
#define EDG_POOL_CASE(NV)                                                                                   \
    rc = opt_in_smem(pool_staged_kernel<T, NV>, smem, &seen[NV - 1]);                                       \
    if (rc) return rc;                                                                                      \
    pool_staged_kernel<T, NV><<<blocks, blk, smem, s>>>((const T*)h, ldh, sent_ptr, row_sent, N, B, D, p.tile_rows,    \
                                                       p.cap_rows, g, pp, aa, v0 == 0 ? hmax : nullptr);
    switch (nv) {
      case 1: EDG_POOL_CASE(1) break;
      default: EDG_POOL_CASE(2) break;
    }
#undef EDG_POOL_CASE
  }
  return check_launch();
}

template <typename T, int I64, int Q>
static int launch_scores_q(const void* h, int64_t ldh, const int32_t* sent_ptr, const int32_t* row_sent, int N, int B, int D,
                           int chunks, const WindowPlan& p, size_t smem, const float* gate, const float* v, const float* c,
                           const void* dist, float* scores, float* kl_b, float* dv_unit, float* dc_unit, float* u_unit, float* sf_unit,
                           cudaStream_t s) {
  static size_t seen = 0;
  int rc = opt_in_smem(scores_staged_kernel<T, I64, Q>, smem, &seen);
  if (rc) return rc;
  const unsigned blocks = (unsigned)((N + p.tile_rows - 1) / p.tile_rows);
  scores_staged_kernel<T, I64, Q><<<blocks, dim3(32, kScoresWarps), smem, s>>>((const T*)h, ldh, sent_ptr, row_sent, N, B, D, chunks,
                                                                   p.tile_rows, p.cap_rows, gate, v, c, dist, scores, kl_b,
                                                                   dv_unit, dc_unit, u_unit, sf_unit);
  return check_launch();
}

template <typename T>
int scores_kl_staged(const void* h, int64_t ldh, const int32_t* sent_ptr, const int32_t* row_sent, int N, int B, int D,
                     int max_len, const float* gate, const float* v, const float* c, const void* dist, int dist_i64,
                     float* scores, float* kl_b, float* dv_unit, float* dc_unit, float* u_unit, float* sf_unit, cudaStream_t s) {
  constexpr int E = Vec16<T>::kElems;
  const int chunks = (D + E - 1) / E;
  if (!row_sent || max_len <= 0 || N <= 0 || chunks > 32 * kSMaxQ || max_len > 32 * kSMaxPass) return 1;
  const size_t wbuf = (size_t)kScoresWarps * chunks * E * sizeof(float);          // per-warp gate*v of the current sentence
  const WindowPlan p = plan_window((size_t)ldh * sizeof(T), max_len, 0, wbuf);
  if (p.tile_rows < 8) return 1;
  const size_t smem = p.smem_rows + wbuf;
  const int Q = (chunks + 31) / 32;
#define EDG_SC(QQ)                                                                                                       \
  return dist_i64 ? launch_scores_q<T, 1, QQ>(h, ldh, sent_ptr, row_sent, N, B, D, chunks, p, smem, gate, v, c, dist, scores, \
                                              kl_b, dv_unit, dc_unit, u_unit, sf_unit, s)                                                 \
                  : launch_scores_q<T, 0, QQ>(h, ldh, sent_ptr, row_sent, N, B, D, chunks, p, smem, gate, v, c, dist, scores, \
                                              kl_b, dv_unit, dc_unit, u_unit, sf_unit, s);
  switch (Q) {
    case 1: EDG_SC(1)
    case 2: EDG_SC(2)
    case 3: EDG_SC(3)
    default: EDG_SC(4)
  }
#undef EDG_SC
}

template <typename T>
int head_bwd_staged(const void* h, int64_t ldh, const int32_t* sent_ptr, const int32_t* row_sent, int N, int B, int D,
                    int max_len, const float* gate, const float* v, const void* dist, int dist_i64, const float* scores,
                    const float* kl_b, const float* g_kl, const float* g_scores, const float* g_pooled, const int32_t* arg,
                    const void* g_xout, int64_t ldgx, void* dh, int64_t lddh, float* dgate, float* dv, float* dc,
                    cudaStream_t s) {
  constexpr int E = Vec16<T>::kElems;
  const int chunks = (D + E - 1) / E;
  if (!row_sent || max_len <= 0 || N <= 0 || chunks > 256) return 1;
  const dim3 blk = chunk_block(chunks);
  const WindowPlan p = plan_window((size_t)ldh * sizeof(T), max_len, 4);
  if (p.tile_rows < 8) return 1;
  {
    const dim3 blk = chunk_block(chunks);
    if (blk.x * blk.y < 32) return 1;              // phase 1 needs one full warp
  }
  const size_t smem = p.smem_rows + (size_t)p.cap_rows * sizeof(float);
  const unsigned blocks = (unsigned)((N + p.tile_rows - 1) / p.tile_rows);
  static size_t seen[2] = {0, 0};
  int rc;
  if (dist_i64) {
    rc = opt_in_smem(head_bwd_staged_kernel<T, 1>, smem, &seen[1]);
    if (rc) return rc;
    head_bwd_staged_kernel<T, 1><<<blocks, chunk_block(chunks), smem, s>>>(
        (const T*)h, ldh, sent_ptr, row_sent, N, B, D, p.tile_rows, p.cap_rows, gate, v, dist, scores, kl_b, g_kl, g_scores,
        g_pooled, arg, (const T*)g_xout, ldgx, (T*)dh, lddh, dgate, dv, dc);
  } else {
    rc = opt_in_smem(head_bwd_staged_kernel<T, 0>, smem, &seen[0]);
    if (rc) return rc;
    head_bwd_staged_kernel<T, 0><<<blocks, chunk_block(chunks), smem, s>>>(
        (const T*)h, ldh, sent_ptr, row_sent, N, B, D, p.tile_rows, p.cap_rows, gate, v, dist, scores, kl_b, g_kl, g_scores,
        g_pooled, arg, (const T*)g_xout, ldgx, (T*)dh, lddh, dgate, dv, dc);
  }
  return check_launch();
}

}  // namespace edg
