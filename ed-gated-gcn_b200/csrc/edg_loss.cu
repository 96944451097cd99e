// The loss on [B,*]-sized data (train.py:121 `criterion(outputs, targets)` = nn.CrossEntropyLoss, train.py:115-118 the
// weighted sum of the loss terms):
//     loss = mean_b ( logsumexp(logits_b) - logits_b[target_b] )
// and its backward, each one launch; every reduction runs in a fixed order.
#include "edg_common.cuh"

namespace edg {

// ---- cross entropy (mean over the rows whose target is not `ignore`) ----------------------------------
// A warp per row (lanes over the classes).  Every block leaves its (loss sum, row count) in `scratch`; the block that
// takes the last ticket adds the partials in block order (deterministic) and writes out[0] = mean loss, out[1] = count.
constexpr int kCeWarps = 8;
__global__ void __launch_bounds__(kCeWarps * 32)
ce_fwd_kernel(const float* __restrict__ lg, int64_t ldl, const int64_t* __restrict__ tgt, int B, int C, int64_t ignore,
              float* __restrict__ out, int* __restrict__ bad, float* __restrict__ scratch, unsigned* __restrict__ ticket) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.x * kCeWarps + warp;
  float loss = 0.f, cnt = 0.f;
  if (b < B) {
    const int64_t t = tgt[b];
    if (t != ignore && (t < 0 || t >= C)) {
      if (lane == 0) atomicOr(bad, 1);
    } else if (t != ignore) {
      const float* row = lg + (int64_t)b * ldl;
      float m = -INFINITY;
      for (int c = lane; c < C; c += 32) m = fmaxf(m, __ldg(row + c));
      m = warp_max(m);
      float se = 0.f;
      for (int c = lane; c < C; c += 32) se += expf(__ldg(row + c) - m);
      se = warp_sum(se);
      loss = (m + logf(se)) - __ldg(row + t);
      cnt = 1.f;
    }
  }
  __shared__ float ws[kCeWarps], wc[kCeWarps];
  __shared__ bool last;
  if (lane == 0) { ws[warp] = loss; wc[warp] = cnt; }
  __syncthreads();
  if (threadIdx.x == 0) {
    float s = 0.f, c = 0.f;
    for (int w = 0; w < kCeWarps; ++w) { s += ws[w]; c += wc[w]; }
    scratch[2 * blockIdx.x] = s;
    scratch[2 * blockIdx.x + 1] = c;
    __threadfence();
    last = atomicAdd(ticket, 1u) == gridDim.x - 1;
  }
  __syncthreads();
  if (!last) return;
  __threadfence();
  // the last block: fixed-order sum of the per-block partials (lane-strided, then a shuffle tree)
  if (warp == 0) {
    float s = 0.f, c = 0.f;
    for (unsigned k = lane; k < gridDim.x; k += 32) { s += __ldcg(scratch + 2 * k); c += __ldcg(scratch + 2 * k + 1); }
    s = warp_sum(s);
    c = warp_sum(c);
    if (lane == 0) { out[0] = c > 0.f ? s / c : 0.f; out[1] = c; *ticket = 0u; }
  }
}

// d logits[b, c] = (softmax(logits_b)[c] - [c == target_b]) * gscale / count   (zero rows for ignored targets)
__global__ void __launch_bounds__(kCeWarps * 32)
ce_bwd_kernel(const float* __restrict__ lg, int64_t ldl, const int64_t* __restrict__ tgt, int B, int C, int64_t ignore,
              const float* __restrict__ gscale, const float* __restrict__ fwd_out, float* __restrict__ dlg, int64_t lddl) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.x * kCeWarps + warp;
  if (b >= B) return;
  const int64_t t = tgt[b];
  float* o = dlg + (int64_t)b * lddl;
  if (t == ignore || t < 0 || t >= C) {
    for (int c = lane; c < C; c += 32) o[c] = 0.f;
    return;
  }
  const float cnt = __ldg(fwd_out + 1);
  const float k = (gscale ? __ldg(gscale) : 1.f) / (cnt > 0.f ? cnt : 1.f);
  const float* row = lg + (int64_t)b * ldl;
  float m = -INFINITY;
  for (int c = lane; c < C; c += 32) m = fmaxf(m, __ldg(row + c));
  m = warp_max(m);
  float se = 0.f;
  for (int c = lane; c < C; c += 32) se += expf(__ldg(row + c) - m);
  se = warp_sum(se);
  const float inv = 1.f / se;
  for (int c = lane; c < C; c += 32) o[c] = (expf(__ldg(row + c) - m) * inv - (c == t ? 1.f : 0.f)) * k;
}

// ---- loss = w0 t0 + w1 t1 + w2 t2 on device scalars (train.py:115-118: CE + gate_w xy + kl_w kl) and its backward ----
__global__ void loss_combine_kernel(const float* __restrict__ t0, const float* __restrict__ t1, const float* __restrict__ t2,
                                    float w0, float w1, float w2, float* __restrict__ out) {
  if (threadIdx.x == 0) out[0] = (t0 ? w0 * t0[0] : 0.f) + (t1 ? w1 * t1[0] : 0.f) + (t2 ? w2 * t2[0] : 0.f);
}
__global__ void loss_combine_bwd_kernel(const float* __restrict__ g, float w0, float w1, float w2, float* __restrict__ out) {
  if (threadIdx.x == 0) {
    const float gg = g ? g[0] : 1.f;
    out[0] = gg * w0; out[1] = gg * w1; out[2] = gg * w2;
  }
}

}  // namespace edg

using namespace edg;

extern "C" int edg_loss_combine(const float* t0, const float* t1, const float* t2, float w0, float w1, float w2, float* out,
                                edg_stream stream) {
  if (!out) return EDG_ERR_ARG;
  loss_combine_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(t0, t1, t2, w0, w1, w2, out);
  return check_launch();
}

extern "C" int edg_loss_combine_bwd(const float* g, float w0, float w1, float w2, float* out3, edg_stream stream) {
  if (!out3) return EDG_ERR_ARG;
  loss_combine_bwd_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(g, w0, w1, w2, out3);
  return check_launch();
}

// out: device float[2] = { mean loss over the counted rows, number of counted rows }; bad: device int[1], set to 1 when a
// target lies outside [0, C) and is not `ignore_index` (the caller decides when to look: no host sync here);
// ws: edg_cross_entropy_workspace(B) bytes, its LAST 4 bytes a ticket counter that must be zero on the first call (the
// kernel leaves it zero)
extern "C" size_t edg_cross_entropy_workspace(int32_t B) {
  const size_t blocks = B > 0 ? ((size_t)B + kCeWarps - 1) / kCeWarps : 1;
  return (2 * blocks + 1) * sizeof(float);
}

extern "C" int edg_cross_entropy_fwd(const float* logits, int64_t ldl, const int64_t* target, int32_t B, int32_t C,
                                     int64_t ignore_index, float* out, int32_t* bad, void* ws, size_t ws_bytes,
                                     edg_stream stream) {
  if (B < 0 || C <= 0 || !out || !bad || !ws) return EDG_ERR_ARG;
  if (B > 0 && (!logits || !target || ldl < C)) return EDG_ERR_ARG;
  if (ws_bytes < edg_cross_entropy_workspace(B)) return EDG_ERR_WORKSPACE;
  const int blocks = B > 0 ? (B + kCeWarps - 1) / kCeWarps : 1;
  float* scratch = (float*)ws;
  unsigned* ticket = (unsigned*)(scratch + 2 * (size_t)blocks);
  ce_fwd_kernel<<<blocks, kCeWarps * 32, 0, (cudaStream_t)stream>>>(logits, ldl, target, B, C, ignore_index, out, bad, scratch,
                                                                    ticket);
  return check_launch();
}

extern "C" int edg_cross_entropy_bwd(const float* logits, int64_t ldl, const int64_t* target, int32_t B, int32_t C,
                                     int64_t ignore_index, const float* gscale, const float* fwd_out, float* dlogits,
                                     int64_t lddl, edg_stream stream) {
  if (B < 0 || C <= 0) return EDG_ERR_ARG;
  if (B == 0) return EDG_OK;
  if (!logits || !target || !fwd_out || !dlogits || ldl < C || lddl < C) return EDG_ERR_ARG;
  ce_bwd_kernel<<<(B + kCeWarps - 1) / kCeWarps, kCeWarps * 32, 0, (cudaStream_t)stream>>>(logits, ldl, target, B, C,
                                                                                         ignore_index, gscale, fwd_out, dlogits,
                                                                                         lddl);
  return check_launch();
}
