// The block's classifier head and the collapsed-scores algebra as one kernel each way (bert_amir5.py:643-646):
//     pooled_b = g_b * hmax_b                     (optional: pooled is an input when the gate is not given)
//     logits_b = W [a_b | pooled_b] + bias        W fp32 [C, 2D] (self.dense)
//     r_b      = Wfc[:, D:] af_b                  af = a, or sigmoid(a) under BertAmir54's fc = Sequential(Sigmoid, Linear)
//     c_b      = logits_b . (r_b + bfc),   v_b = logits_b^T Wfc[:, :D]
// and its backward, with u_b = [s dv_b | s dc_b af_b]:
//     dlg_b = g_logits_b + Wfc u_b + s dc_b bfc
//     da_b  = s dc_b (logits_b^T Wfc[:, D:]) (* af (1 - af) under fc_sigmoid) + dlg_b^T W[:, :D]
//     dp_b  = dlg_b^T W[:, D:] + g_pooled_b
// Either head may be left out (template flags HEAD / FC): without the dense head (a torch logits_fn) the logits are an
// input and only the fc terms are formed; without fc (a DenseHead called on its own) only the logits and their input
// gradients are.  A block owns 8 sentences and both column halves, so v, c and the input gradients follow the logits
// without leaving the SM.  [B,*] work is bound by latency and by how many blocks carry it, not by bytes (DESIGN
// section 5): 512 blocks of 128 threads at C2, all resident at once.
//
// Every sum has a fixed fp32 order (lane-strided fmaf chains closed by an xor butterfly for the K = D reductions,
// classes in ascending order for the K = C products, sentences in blocks of 32 then blocks in order for the parameter
// gradients), and the order of each sum is the same whichever heads a launch runs: the combined launch gives the bits
// of the dense-only and fc-only launches composed.  A torch-head and a DenseHead training run therefore follow the same
// arithmetic -- which matters here: d kl / d c is zero analytically (the softmax over a sentence's scores does not see
// a shift), so d fc.bias is pure rounding, and Adam turns any reordering of it into different parameters.
// Phase 1 (the K = D reductions) stages the pass's rows in shared memory and reads the weights through L1; a warp
// takes 4 sentences x 8 classes and reduces the 32 lane-partial sums in one scattering butterfly.  Phase 2 (the K = C
// products) reads the weights through L1 with 128-bit loads, a thread owning 4 sentences x 4 columns.  The parameter
// gradients (edg_block_head_wgrad) are one partial launch plus one reduction in block order.
#include "edg_common.cuh"

namespace edg {

constexpr int kHeadMaxC = 64;
constexpr int kHeadGraphs = 32;           // sentences per block (parameter-gradient kernel)
constexpr int kHeadThreads = 256;
constexpr int kHeadPitch = 320;           // columns staged per pass (compile-time: shared-memory offsets become immediates)
constexpr int kBhS = 8;                   // sentences per block (forward / input-gradient kernels)
constexpr int kBhWarps = 4;
constexpr int kBhThreads = 32 * kBhWarps;
constexpr int kBhP = kHeadPitch;          // columns per phase-1 pass (a multiple of 32: lane residues stay aligned)

// rows [b0, b0 + nb) of x[:, col0 : col0 + lim) into Xs[kBhS][kBhP] (zero beyond nb / lim), each element times m[., .]
// when m is given (the product is also written to `out` [B, ldo] when given) or times rs[row] when rs is given -- one
// rounding per product, as in the torch product gate * hmax
template <bool VEC>
__device__ __forceinline__ void bh_stage_rows(float* __restrict__ Xs, const float* __restrict__ x, int64_t ldx,
                                              const float* __restrict__ m, int64_t ldm, float* __restrict__ out,
                                              int64_t ldo, const float* rs, int b0, int nb, int col0, int lim) {
  if (VEC) {
    constexpr int P4 = kBhP / 4;
#pragma unroll 4
    for (int i = threadIdx.x; i < kBhS * P4; i += kBhThreads) {
      const int s = i / P4, k = (i - s * P4) * 4;
      float4 u = make_float4(0.f, 0.f, 0.f, 0.f);
      if (s < nb && k < lim) {
        const int64_t b = b0 + s;
        u = __ldg(reinterpret_cast<const float4*>(x + b * ldx + col0 + k));
        if (m) {
          const float4 g = __ldg(reinterpret_cast<const float4*>(m + b * ldm + col0 + k));
          u.x *= g.x; u.y *= g.y; u.z *= g.z; u.w *= g.w;
          if (out) *reinterpret_cast<float4*>(out + b * ldo + col0 + k) = u;
        }
        if (rs) { const float r = rs[s]; u.x *= r; u.y *= r; u.z *= r; u.w *= r; }
      }
      *reinterpret_cast<float4*>(Xs + s * kBhP + k) = u;
    }
  } else {
#pragma unroll 4
    for (int i = threadIdx.x; i < kBhS * kBhP; i += kBhThreads) {
      const int s = i / kBhP, k = i - s * kBhP;
      float u = 0.f;
      if (s < nb && k < lim) {
        const int64_t b = b0 + s;
        u = __ldg(x + b * ldx + col0 + k);
        if (m) {
          u *= __ldg(m + b * ldm + col0 + k);
          if (out) out[b * ldo + col0 + k] = u;
        }
        if (rs) u *= rs[s];
      }
      Xs[i] = u;
    }
  }
}

// Phase 1 of one pass: for both halves h (rows Xs[h] against W[:, wcol[h] + d0 + .]), every sentence and class,
//     out[h][s][c] += warp_sum over lanes r of ( sum over the pass columns jj = r, r + 32, ... of x[s][jj] W[c][jj] )
// (lane-strided fmaf chains, xor-butterfly across the lanes).  A warp takes 4 sentences x 8 classes at a time (every
// staged x and every W element loaded feeds 8 or 4 fmas) and reduces those 32 sums in one xor-butterfly that scatters
// them over the lanes: 31 shuffles instead of 32 x 5, with each sum built from the same pairs as warp_sum's.
template <int NCG8>
__device__ __forceinline__ void bh_pass(const float* __restrict__ Xs, const float* __restrict__ W, int64_t ldw,
                                        int wcol0, int wcol1, int d0, int lim, int C, float* __restrict__ out) {
  constexpr int G = 2 * (kBhS / 4) * NCG8;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int gi = warp; gi < G; gi += kBhWarps) {
    const int h = gi / ((kBhS / 4) * NCG8), rem = gi - h * ((kBhS / 4) * NCG8);
    const int sg = rem / NCG8, cg = rem - sg * NCG8;
    const float* xr = Xs + (h * kBhS + 4 * sg) * kBhP;
    const float* wr[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) wr[j] = W + (int64_t)min(8 * cg + j, C - 1) * ldw + (h ? wcol1 : wcol0) + d0;
    float v[32];
#pragma unroll
    for (int o = 0; o < 32; ++o) v[o] = 0.f;
#pragma unroll 2
    for (int jj = lane; jj < lim; jj += 32) {
      float x[4], w[8];
#pragma unroll
      for (int i = 0; i < 4; ++i) x[i] = xr[i * kBhP + jj];
#pragma unroll
      for (int j = 0; j < 8; ++j) w[j] = __ldg(wr[j] + jj);
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) v[i * 8 + j] = fmaf(x[i], w[j], v[i * 8 + j]);
    }
    // lane L ends with sum L (sentence 4 sg + L / 8, class 8 cg + L % 8)
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) {
      const bool up = (lane & off) != 0;
#pragma unroll
      for (int o = 0; o < off; ++o) {
        const float send = up ? v[o] : v[o + off];
        const float keep = up ? v[o + off] : v[o];
        v[o] = keep + __shfl_xor_sync(0xffffffffu, send, off);
      }
    }
    const int s = 4 * sg + (lane >> 3), c = 8 * cg + (lane & 7);
    if (c < C) out[(h * kBhS + s) * (8 * NCG8) + c] += v[0];
  }
}

// phase 2: out[s][j] = sum_c coef[c][s] Wm[c][j] for the block's sentences, column quads (VEC) or columns; `epi(s, j,
// acc)` receives 4 sentences x 4 columns (VEC; s, j = first of each) or 4 sentences x 1 column.  Fixed order over c.
template <int CP, bool VEC, class Epi>
__device__ __forceinline__ void bh_mix(const float (*coef)[kBhS], const float* __restrict__ Wm, int64_t ldw, int C,
                                       int D, int nb, Epi epi) {
  constexpr int SG = kBhS / 4;
  const int ncol = VEC ? D / 4 : D;
  for (int it = threadIdx.x; it < ncol * SG; it += kBhThreads) {
    const int jc = it % ncol, s0 = (it / ncol) * 4;
    if (s0 >= nb) continue;
    if (VEC) {
      float acc[4][4] = {};
      const float* wp = Wm + 4 * jc;
#pragma unroll 4
      for (int c = 0; c < C; ++c) {
        const float4 w = __ldg(reinterpret_cast<const float4*>(wp + (int64_t)c * ldw));
        const float4 l = *reinterpret_cast<const float4*>(&coef[c][s0]);
        const float lv[4] = {l.x, l.y, l.z, l.w};
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          acc[i][0] = fmaf(lv[i], w.x, acc[i][0]); acc[i][1] = fmaf(lv[i], w.y, acc[i][1]);
          acc[i][2] = fmaf(lv[i], w.z, acc[i][2]); acc[i][3] = fmaf(lv[i], w.w, acc[i][3]);
        }
      }
      epi(s0, 4 * jc, acc);
    } else {
      float acc[4][4] = {};
      for (int c = 0; c < C; ++c) {
        const float w = __ldg(Wm + (int64_t)c * ldw + jc);
        const float4 l = *reinterpret_cast<const float4*>(&coef[c][s0]);
        acc[0][0] = fmaf(l.x, w, acc[0][0]); acc[1][0] = fmaf(l.y, w, acc[1][0]);
        acc[2][0] = fmaf(l.z, w, acc[2][0]); acc[3][0] = fmaf(l.w, w, acc[3][0]);
      }
      epi(s0, jc, acc);
    }
  }
}

// ---- forward ----------------------------------------------------------------------------------------------------
// HEAD: the logits from [a | pooled] (else read from `logits`); FC: v and c from the logits.
template <int NCG8, bool VEC, bool HEAD, bool FC>
__global__ void __launch_bounds__(kBhThreads, 4)
block_head_fwd_kernel(const float* __restrict__ a, int64_t lda, const float* __restrict__ af, int64_t ldf,
                      const float* __restrict__ p, int64_t ldp, const float* __restrict__ g, int64_t ldg,
                      const float* __restrict__ W, int64_t ldw, const float* __restrict__ bias,
                      const float* __restrict__ Wf, int64_t ldfw, const float* __restrict__ bf, int B, int D, int C,
                      float* __restrict__ pooled, float* __restrict__ logits, float* __restrict__ v,
                      float* __restrict__ cout) {
  constexpr int CP = 8 * NCG8;
  __shared__ __align__(16) float Xs[2 * kBhS * kBhP];                  // a | pooled rows of the pass; then va
  __shared__ float part[2 * kBhS * CP];                                 // W[:, :D] a  |  W[:, D:] pooled
  __shared__ __align__(16) float lg_t[CP][kBhS];                       // logits [class][sentence]
  const int b0 = blockIdx.x * kBhS;
  const int nb = min(kBhS, B - b0);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if constexpr (HEAD) {
    for (int i = threadIdx.x; i < 2 * kBhS * CP; i += kBhThreads) part[i] = 0.f;
    for (int d0 = 0; d0 < D; d0 += kBhP) {
      const int lim = min(kBhP, D - d0);
      __syncthreads();                                                   // previous pass consumed (part zeroed)
      bh_stage_rows<VEC>(Xs, a, lda, nullptr, 0, nullptr, 0, nullptr, b0, nb, d0, lim);
      bh_stage_rows<VEC>(Xs + kBhS * kBhP, p, ldp, g, ldg, pooled, D, nullptr, b0, nb, d0, lim);
      __syncthreads();
      bh_pass<NCG8>(Xs, W, ldw, 0, D, d0, lim, C, part);
    }
    __syncthreads();
  }
  // logits = (W[:, :D] a + bias) + W[:, D:] pooled
  for (int i = threadIdx.x; i < kBhS * CP; i += kBhThreads) {
    const int s = i / CP, c = i - s * CP;
    float l = 0.f;
    if (s < nb && c < C) {
      if constexpr (HEAD) {
        l = (part[s * CP + c] + (bias ? __ldg(bias + c) : 0.f)) + part[(kBhS + s) * CP + c];
        logits[(int64_t)(b0 + s) * C + c] = l;
      } else {
        l = __ldg(logits + (int64_t)(b0 + s) * C + c);
      }
    }
    lg_t[c][s] = l;
  }
  if constexpr (!FC) return;
  __syncthreads();
  // v = logits^T Wfc[:, :D]
  bh_mix<CP, VEC>(lg_t, Wf, ldfw, C, D, nb, [&](int s0, int j, const float (&o)[4][4]) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      if (s0 + i >= nb) break;
      float* dst = v + (int64_t)(b0 + s0 + i) * D + j;
      if (VEC) *reinterpret_cast<float4*>(dst) = make_float4(o[i][0], o[i][1], o[i][2], o[i][3]);
      else *dst = o[i][0];
    }
  });
  // c = warp_sum over lanes of (sum over d = lane, lane + 32, ... of af[d] va[d]) + logits . bfc, va = logits^T
  // Wfc[:, D:]; va goes through shared memory a pass at a time, a warp owns 2 sentences
  float* va = Xs;                                                        // [kBhS][kBhP]
  float cacc[2] = {0.f, 0.f};
  for (int d0 = 0; d0 < D; d0 += kBhP) {
    const int lim = min(kBhP, D - d0);
    __syncthreads();
    bh_mix<CP, VEC>(lg_t, Wf + D + d0, ldfw, C, lim, nb, [&](int s0, int j, const float (&o)[4][4]) {
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        if (VEC) *reinterpret_cast<float4*>(va + (s0 + i) * kBhP + j) = make_float4(o[i][0], o[i][1], o[i][2], o[i][3]);
        else va[(s0 + i) * kBhP + j] = o[i][0];
      }
    });
    __syncthreads();
#pragma unroll
    for (int q = 0; q < 2; ++q) {
      const int s = 2 * warp + q;
      if (s >= nb) break;
      for (int jj = lane; jj < lim; jj += 32)
        cacc[q] = fmaf(__ldg(af + (int64_t)(b0 + s) * ldf + d0 + jj), va[s * kBhP + jj], cacc[q]);
    }
  }
#pragma unroll
  for (int q = 0; q < 2; ++q) {
    const int s = 2 * warp + q;
    if (s >= nb) break;
    float t = warp_sum(cacc[q]);
    if (lane == 0) {
      for (int c = 0; c < C; ++c) t = fmaf(lg_t[c][s], __ldg(bf + c), t);
      cout[b0 + s] = t;
    }
  }
}

// ---- input gradients -----------------------------------------------------------------------------------------------
// dlg = g + ((Wfc[:, :D] (s dv) + s dc bfc) + Wfc[:, D:] (s dc af)), da = dlg^T W[:, :D] + (s dc) (logits^T Wfc[:, D:]),
// dp = dlg^T W[:, D:] + g_pooled.  FC: the fc terms (when dv is given); HEAD: the dense head's terms and dp.
template <int NCG8, bool VEC, bool HEAD, bool FC>
__global__ void __launch_bounds__(kBhThreads, 4)
block_head_bwd_kernel(const float* __restrict__ lg, const float* __restrict__ a, int64_t lda,
                      const float* __restrict__ af, int64_t ldf, int fc_sigmoid, const float* __restrict__ W, int64_t ldw,
                      const float* __restrict__ Wf, int64_t ldfw, const float* __restrict__ bf,
                      const float* __restrict__ dv, const float* __restrict__ dc, const float* __restrict__ scale,
                      const float* __restrict__ g_lg, const float* __restrict__ g_p, int B, int D, int C,
                      float* __restrict__ dlg, float* __restrict__ da, float* __restrict__ dp) {
  constexpr int CP = 8 * NCG8;
  __shared__ __align__(16) float Xs[2 * kBhS * kBhP];                  // s dv | s dc af rows of the pass
  __shared__ float part[2 * kBhS * CP];
  __shared__ __align__(16) float dlg_t[CP][kBhS];                      // d logits [class][sentence]
  __shared__ __align__(16) float lg_t[CP][kBhS];                       // logits   [class][sentence]
  __shared__ float rs_v[kBhS], dc_s[kBhS];
  const int b0 = blockIdx.x * kBhS;
  const int nb = min(kBhS, B - b0);
  const bool scores = FC && dv != nullptr;
  const float sc = (scores && scale) ? __ldg(scale) : 1.f;
  if (threadIdx.x < kBhS) {
    const int s = threadIdx.x;
    rs_v[s] = sc;
    dc_s[s] = (scores && s < nb) ? sc * __ldg(dc + b0 + s) : 0.f;
  }
  for (int i = threadIdx.x; i < 2 * kBhS * CP; i += kBhThreads) part[i] = 0.f;
  for (int d0 = 0; scores && d0 < D; d0 += kBhP) {
    const int lim = min(kBhP, D - d0);
    __syncthreads();
    bh_stage_rows<VEC>(Xs, dv, D, nullptr, 0, nullptr, 0, rs_v, b0, nb, d0, lim);
    bh_stage_rows<VEC>(Xs + kBhS * kBhP, af, ldf, nullptr, 0, nullptr, 0, dc_s, b0, nb, d0, lim);
    __syncthreads();
    bh_pass<NCG8>(Xs, Wf, ldfw, 0, D, d0, lim, C, part);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < kBhS * CP; i += kBhThreads) {
    const int s = i / CP, c = i - s * CP;
    float d = 0.f, l = 0.f;
    if (s < nb && c < C) {
      const int64_t o = (int64_t)(b0 + s) * C + c;
      if (FC) l = __ldg(lg + o);
      if (scores) {
        d = fmaf(dc_s[s], __ldg(bf + c), part[s * CP + c]) + part[(kBhS + s) * CP + c];
        if (g_lg) d = __ldg(g_lg + o) + d;
      } else if (g_lg) {
        d = __ldg(g_lg + o);
      }
      dlg[o] = d;
    }
    dlg_t[c][s] = d;
    lg_t[c][s] = l;
  }
  __syncthreads();
  // d a
  constexpr int SG = kBhS / 4;
  const int ncol = VEC ? D / 4 : D;
  for (int it = threadIdx.x; it < ncol * SG; it += kBhThreads) {
    const int jc = it % ncol, s0 = (it / ncol) * 4;
    if (s0 >= nb) continue;
    const int j = VEC ? 4 * jc : jc;
    const int nj = VEC ? 4 : 1;
    float t1[4][4] = {}, t2[4][4] = {};
#pragma unroll 4
    for (int c = 0; c < C; ++c) {
      float w1[4] = {}, w2[4] = {};
      if (VEC) {
        if (FC) {
          const float4 x = __ldg(reinterpret_cast<const float4*>(Wf + (int64_t)c * ldfw + D + j));
          w1[0] = x.x; w1[1] = x.y; w1[2] = x.z; w1[3] = x.w;
        }
        if (HEAD) {
          const float4 y = __ldg(reinterpret_cast<const float4*>(W + (int64_t)c * ldw + j));
          w2[0] = y.x; w2[1] = y.y; w2[2] = y.z; w2[3] = y.w;
        }
      } else {
        if (FC) w1[0] = __ldg(Wf + (int64_t)c * ldfw + D + j);
        if (HEAD) w2[0] = __ldg(W + (int64_t)c * ldw + j);
      }
      const float4 k = *reinterpret_cast<const float4*>(&lg_t[c][s0]);
      const float4 d = *reinterpret_cast<const float4*>(&dlg_t[c][s0]);
      const float kv[4] = {k.x, k.y, k.z, k.w}, dvv[4] = {d.x, d.y, d.z, d.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          t1[i][q] = fmaf(kv[i], w1[q], t1[i][q]);
          t2[i][q] = fmaf(dvv[i], w2[q], t2[i][q]);
        }
    }
    for (int i = 0; i < 4 && s0 + i < nb; ++i) {
      const int64_t b = b0 + s0 + i;
      float o[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        o[q] = HEAD ? t2[i][q] : 0.f;
        if (scores && q < nj) {
          float f = dc_s[s0 + i] * t1[i][q];
          if (fc_sigmoid) {
            const float z = __ldg(af + b * ldf + j + q);
            f = (f * z) * (1.f - z);
          }
          o[q] = HEAD ? o[q] + f : f;
        }
      }
      float* dst = da + b * D + j;
      if (VEC) *reinterpret_cast<float4*>(dst) = make_float4(o[0], o[1], o[2], o[3]);
      else *dst = o[0];
    }
  }
  // d p = dlg^T W[:, D:] + g_pooled
  if constexpr (HEAD) bh_mix<CP, VEC>(dlg_t, W + D, ldw, C, D, nb, [&](int s0, int j, const float (&o)[4][4]) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      if (s0 + i >= nb) break;
      const int64_t off = (int64_t)(b0 + s0 + i) * D + j;
      if (VEC) {
        float4 r = make_float4(o[i][0], o[i][1], o[i][2], o[i][3]);
        if (g_p) {
          const float4 q = __ldg(reinterpret_cast<const float4*>(g_p + off));
          r.x += q.x; r.y += q.y; r.z += q.z; r.w += q.w;
        }
        *reinterpret_cast<float4*>(dp + off) = r;
      } else {
        dp[off] = o[i][0] + (g_p ? __ldg(g_p + off) : 0.f);
      }
    }
  });
}

// rows [b0, b0+nb) of x[:, d0 : d0+kHeadPitch) into Xs [32][kHeadPitch], zero beyond nb / lim
__device__ __forceinline__ void stage_rows_chunk(float* __restrict__ Xs, const float* __restrict__ x, int64_t ldx, int b0,
                                                 int nb, int d0, int lim, bool vec4) {
  if (vec4) {
    constexpr int P4 = kHeadPitch / 4;
#pragma unroll 4
    for (int i = threadIdx.x; i < kHeadGraphs * P4; i += kHeadThreads) {
      const int g = i / P4, jj = (i - g * P4) << 2;
      float4 u = make_float4(0.f, 0.f, 0.f, 0.f);
      if (g < nb && jj < lim) u = __ldg(reinterpret_cast<const float4*>(x + (int64_t)(b0 + g) * ldx + d0 + jj));
      *reinterpret_cast<float4*>(Xs + g * kHeadPitch + jj) = u;
    }
  } else {
#pragma unroll 4
    for (int i = threadIdx.x; i < kHeadGraphs * kHeadPitch; i += kHeadThreads) {
      const int g = i / kHeadPitch, jj = i - g * kHeadPitch;
      Xs[i] = (g < nb && jj < lim) ? __ldg(x + (int64_t)(b0 + g) * ldx + d0 + jj) : 0.f;
    }
  }
}

// ---- parameter gradients: per-block partials [nblocks][C][4D + 2] -----------------------------------------------
// Block (x, q): 32 sentences x column quarter q of [d Wfc | d W]:  q = 0: logits^T (s dv),  q = 1: logits^T (s dc af)
// (+ d bfc = logits^T (s dc), column 4D),  q = 2: dlg^T a,  q = 3: dlg^T pooled (+ d bias = colsum dlg, column 4D + 1).
// Quarters 0-1 run when the scores carry gradient (dv given), quarters 2-3 when dlg is given.
template <int CP>
__global__ void __launch_bounds__(kHeadThreads, 2)
block_head_wgrad_kernel(const float* __restrict__ lg, const float* __restrict__ dlg, const float* __restrict__ a,
                        int64_t lda, const float* __restrict__ af, int64_t ldf, const float* __restrict__ p, int64_t ldp,
                        const float* __restrict__ dv, const float* __restrict__ dc, const float* __restrict__ scale,
                        int B, int D, int C, int vec4, float* __restrict__ partial) {
  extern __shared__ __align__(16) float head_smem[];
  __shared__ __align__(16) float k_s[kHeadGraphs][CP];                  // coefficient rows [sentence][class]
  __shared__ float rs[kHeadGraphs];
  float* Xs = head_smem;                                                 // [32][kHeadPitch]
  const int q = blockIdx.y;
  const bool fc = q < 2;
  if (fc ? dv == nullptr : dlg == nullptr) return;
  const int b0 = blockIdx.x * kHeadGraphs;
  const int nb = min(kHeadGraphs, B - b0);
  const float sc = (fc && scale) ? __ldg(scale) : 1.f;
  const float* coef = fc ? lg : dlg;
  for (int i = threadIdx.x; i < kHeadGraphs * CP; i += kHeadThreads) {
    const int s = i / CP, c = i - s * CP;
    k_s[s][c] = (s < nb && c < C) ? __ldg(coef + (int64_t)(b0 + s) * C + c) : 0.f;
  }
  if (threadIdx.x < kHeadGraphs) {
    const int s = threadIdx.x;
    rs[s] = s >= nb ? 0.f : q == 0 ? sc : q == 1 ? sc * __ldg(dc + b0 + s) : 1.f;
  }
  const float* x = q == 0 ? dv : q == 1 ? af : q == 2 ? a : p;
  const int64_t ldx = q == 0 ? D : q == 1 ? ldf : q == 2 ? lda : ldp;
  const int W4 = 4 * D + 2;
  float* P = partial + (int64_t)blockIdx.x * C * W4;
  for (int d0 = 0; d0 < D; d0 += kHeadPitch) {
    __syncthreads();
    const int lim = min(kHeadPitch, D - d0);
    stage_rows_chunk(Xs, x, ldx, b0, nb, d0, lim, vec4 != 0);
    __syncthreads();
    for (int jj = threadIdx.x; jj < lim; jj += kHeadThreads) {          // thread = column of the pass
      float acc[CP];
#pragma unroll
      for (int cc = 0; cc < CP; ++cc) acc[cc] = 0.f;
      const float* ucol = Xs + jj;
#pragma unroll 2
      for (int s = 0; s < kHeadGraphs; ++s) {                           // rows >= nb are zero
        const float u = ucol[s * kHeadPitch] * rs[s];
#pragma unroll
        for (int c4 = 0; c4 < CP; c4 += 4) {
          const float4 l = *reinterpret_cast<const float4*>(&k_s[s][c4]);
          acc[c4] = fmaf(l.x, u, acc[c4]); acc[c4 + 1] = fmaf(l.y, u, acc[c4 + 1]);
          acc[c4 + 2] = fmaf(l.z, u, acc[c4 + 2]); acc[c4 + 3] = fmaf(l.w, u, acc[c4 + 3]);
        }
      }
      float* pc = P + q * D + d0 + jj;
#pragma unroll
      for (int cc = 0; cc < CP; ++cc)
        if (cc < C) pc[(int64_t)cc * W4] = acc[cc];
    }
  }
  if ((q == 1 || q == 3) && threadIdx.x < C) {                          // bias columns
    float t = 0.f;
    for (int s = 0; s < nb; ++s) t = fmaf(rs[s], k_s[s][threadIdx.x], t);
    P[(int64_t)threadIdx.x * W4 + 4 * D + (q == 1 ? 0 : 1)] = t;
  }
}

// sum of the per-block partials in block order -> d Wfc [C, 2D], d W [C, 2D], d bfc [C], d bias [C] (each when present)
__global__ void __launch_bounds__(256)
block_head_wgrad_reduce_kernel(const float* __restrict__ partial, int nblocks, int C, int D, int fc, int head,
                               float* __restrict__ dWf, float* __restrict__ dbf, float* __restrict__ dW,
                               float* __restrict__ db) {
  const int W4 = 4 * D + 2;
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t per = (int64_t)C * W4;
  if (idx >= per) return;
  const int cc = (int)(idx / W4), j = (int)(idx - (int64_t)cc * W4);
  const bool is_fc = j < 2 * D || j == 4 * D;
  if (is_fc ? !fc : !head) return;
  float* dst;
  if (j < 2 * D) dst = dWf + (int64_t)cc * 2 * D + j;
  else if (j < 4 * D) dst = dW + (int64_t)cc * 2 * D + (j - 2 * D);
  else if (j == 4 * D) dst = dbf + cc;
  else if (db) dst = db + cc;
  else return;
  float s = 0.f;
#pragma unroll 8
  for (int k = 0; k < nblocks; ++k) s += partial[k * per + idx];
  *dst = s;
}

// the instantiation for C, the row alignment and the heads present (at least one)
template <bool HEAD, bool FC, class Launch>
int bh_fwd_launch(int C, bool vec4, Launch launch) {
  if (C <= 8) return vec4 ? launch(block_head_fwd_kernel<1, true, HEAD, FC>) : launch(block_head_fwd_kernel<1, false, HEAD, FC>);
  if (C <= 40) return vec4 ? launch(block_head_fwd_kernel<5, true, HEAD, FC>) : launch(block_head_fwd_kernel<5, false, HEAD, FC>);
  return vec4 ? launch(block_head_fwd_kernel<8, true, HEAD, FC>) : launch(block_head_fwd_kernel<8, false, HEAD, FC>);
}

template <bool HEAD, bool FC, class Launch>
int bh_bwd_launch(int C, bool vec4, Launch launch) {
  if (C <= 8) return vec4 ? launch(block_head_bwd_kernel<1, true, HEAD, FC>) : launch(block_head_bwd_kernel<1, false, HEAD, FC>);
  if (C <= 40) return vec4 ? launch(block_head_bwd_kernel<5, true, HEAD, FC>) : launch(block_head_bwd_kernel<5, false, HEAD, FC>);
  return vec4 ? launch(block_head_bwd_kernel<8, true, HEAD, FC>) : launch(block_head_bwd_kernel<8, false, HEAD, FC>);
}

}  // namespace edg

using namespace edg;

extern "C" int edg_block_head_fwd(const float* a, int64_t lda, const float* a_fc, int64_t ldf, const float* p,
                                  int64_t ldp, const float* g, int64_t ldg, const float* W, int64_t ldw,
                                  const float* bias, const float* fc_w, int64_t ldfw, const float* fc_b, int32_t B,
                                  int32_t D, int32_t C, float* pooled, float* logits, float* v, float* c,
                                  edg_stream stream) {
  const bool head = W != nullptr, fc = fc_w != nullptr;
  if (B < 0 || D <= 0 || C <= 0 || (!head && !fc)) return EDG_ERR_ARG;
  if (C > kHeadMaxC) return EDG_ERR_UNSUPPORTED;
  if (B == 0) return EDG_OK;
  if (!logits || (head && (!a || !p || (g && !pooled))) || (fc && (!a_fc || !fc_b || !v || !c))) return EDG_ERR_ARG;
  if ((head && (lda < D || ldp < D || (g && ldg < D) || ldw < 2 * D)) || (fc && (ldf < D || ldfw < 2 * D)))
    return EDG_ERR_ARG;
  const bool vec4 = (D & 3) == 0 && (lda & 3) == 0 && (ldf & 3) == 0 && (ldp & 3) == 0 && (ldg & 3) == 0 &&
                    (ldw & 3) == 0 && (ldfw & 3) == 0 && aligned16(a) && aligned16(a_fc) && aligned16(p) &&
                    aligned16(g) && aligned16(W) && aligned16(fc_w) && aligned16(pooled) && aligned16(v);
  const unsigned blocks = (unsigned)((B + kBhS - 1) / kBhS);
  cudaStream_t s = (cudaStream_t)stream;
  auto launch = [&](auto kern) -> int {
    kern<<<blocks, kBhThreads, 0, s>>>(a, lda, a_fc, ldf, p, ldp, g, ldg, W, ldw, bias, fc_w, ldfw, fc_b, B, D, C, pooled,
                                       logits, v, c);
    return check_launch();
  };
  if (!head) return bh_fwd_launch<false, true>(C, vec4, launch);
  if (!fc) return bh_fwd_launch<true, false>(C, vec4, launch);
  return bh_fwd_launch<true, true>(C, vec4, launch);
}

extern "C" int edg_block_head_bwd(const float* logits, const float* a, int64_t lda, const float* a_fc, int64_t ldf,
                                  int fc_sigmoid, const float* W, int64_t ldw, const float* fc_w, int64_t ldfw,
                                  const float* fc_b, const float* dv, const float* dc, const float* scale,
                                  const float* g_logits, const float* g_pooled, int32_t B, int32_t D, int32_t C,
                                  float* dlg, float* da, float* dp, edg_stream stream) {
  const bool head = W != nullptr, fc = fc_w != nullptr;
  if (B < 0 || D <= 0 || C <= 0 || (!head && !fc)) return EDG_ERR_ARG;
  if (C > kHeadMaxC) return EDG_ERR_UNSUPPORTED;
  if (B == 0) return EDG_OK;
  if (!a || !dlg || !da || (head && !dp) || (!dv) != (!dc) || (!fc && dv)) return EDG_ERR_ARG;
  if (fc && (!logits || !a_fc || !fc_b)) return EDG_ERR_ARG;
  if (lda < D || (head && ldw < 2 * D) || (fc && (ldf < D || ldfw < 2 * D))) return EDG_ERR_ARG;
  const bool vec4 = (D & 3) == 0 && (lda & 3) == 0 && (ldf & 3) == 0 && (ldw & 3) == 0 && (ldfw & 3) == 0 &&
                    aligned16(a) && aligned16(a_fc) && aligned16(W) && aligned16(fc_w) && aligned16(dv) &&
                    aligned16(g_pooled) && aligned16(da) && aligned16(dp);
  const unsigned blocks = (unsigned)((B + kBhS - 1) / kBhS);
  cudaStream_t s = (cudaStream_t)stream;
  auto launch = [&](auto kern) -> int {
    kern<<<blocks, kBhThreads, 0, s>>>(logits, a, lda, a_fc, ldf, fc_sigmoid, W, ldw, fc_w, ldfw, fc_b, dv, dc, scale,
                                       g_logits, g_pooled, B, D, C, dlg, da, dp);
    return check_launch();
  };
  if (!head) return bh_bwd_launch<false, true>(C, vec4, launch);
  if (!fc) return bh_bwd_launch<true, false>(C, vec4, launch);
  return bh_bwd_launch<true, true>(C, vec4, launch);
}

extern "C" size_t edg_block_head_wgrad_workspace(int32_t B, int32_t D, int32_t C) {
  if (B <= 0 || D <= 0 || C <= 0) return 16;
  const size_t blocks = (size_t)(B + kHeadGraphs - 1) / kHeadGraphs;
  return blocks * (size_t)C * (4 * (size_t)D + 2) * sizeof(float);
}

extern "C" int edg_block_head_wgrad(const float* logits, const float* dlg, const float* a, int64_t lda, const float* a_fc,
                                    int64_t ldf, const float* pooled, int64_t ldp, const float* dv, const float* dc,
                                    const float* scale, int32_t B, int32_t D, int32_t C, float* dW, float* dbias,
                                    float* d_fc_w, float* d_fc_b, void* ws, size_t ws_bytes, edg_stream stream) {
  if (B < 0 || D <= 0 || C <= 0 || (!dv) != (!dc)) return EDG_ERR_ARG;
  if (C > kHeadMaxC) return EDG_ERR_UNSUPPORTED;
  const bool fc = dv != nullptr, head = dlg != nullptr;
  if (fc && (!d_fc_w || !d_fc_b)) return EDG_ERR_ARG;
  if (head && !dW) return EDG_ERR_ARG;
  cudaStream_t s = (cudaStream_t)stream;
  if (B == 0) {
    if (fc) {
      cudaMemsetAsync(d_fc_w, 0, (size_t)C * 2 * D * sizeof(float), s);
      cudaMemsetAsync(d_fc_b, 0, C * sizeof(float), s);
    }
    if (head) {
      cudaMemsetAsync(dW, 0, (size_t)C * 2 * D * sizeof(float), s);
      if (dbias) cudaMemsetAsync(dbias, 0, C * sizeof(float), s);
    }
    return check_launch();
  }
  if (!fc && !head) return EDG_OK;
  if (!ws || (fc && (!logits || !a_fc)) || (head && (!a || !pooled))) return EDG_ERR_ARG;
  if ((head && (lda < D || ldp < D)) || (fc && ldf < D)) return EDG_ERR_ARG;
  if (ws_bytes < edg_block_head_wgrad_workspace(B, D, C)) return EDG_ERR_WORKSPACE;
  const int vec4 = ((D & 3) == 0 && (lda & 3) == 0 && (ldf & 3) == 0 && (ldp & 3) == 0 && aligned16(a) &&
                    aligned16(a_fc) && aligned16(pooled) && aligned16(dv)) ? 1 : 0;
  const int blocks = (B + kHeadGraphs - 1) / kHeadGraphs;
  float* partial = reinterpret_cast<float*>(ws);
  auto launch = [&](auto kern) -> int {
    const size_t smem = (size_t)kHeadGraphs * kHeadPitch * sizeof(float);
    if (int rc_ = ensure_dyn_smem((const void*)kern, smem)) return rc_;
    kern<<<dim3(blocks, 4), kHeadThreads, smem, s>>>(logits, dlg, a, lda, a_fc, ldf, pooled, ldp, dv, dc, scale, B, D, C,
                                                     vec4, partial);
    return check_launch();
  };
  int rc;
  if (C <= 8) rc = launch(block_head_wgrad_kernel<8>);
  else if (C <= 36) rc = launch(block_head_wgrad_kernel<36>);
  else rc = launch(block_head_wgrad_kernel<64>);
  if (rc) return rc;
  const int64_t per = (int64_t)C * (4 * D + 2);
  block_head_wgrad_reduce_kernel<<<(unsigned)((per + 255) / 256), 256, 0, s>>>(partial, blocks, C, D, fc ? 1 : 0,
                                                                              head ? 1 : 0, d_fc_w, d_fc_b, dW, dbias);
  return check_launch();
}
