// Integer kernels: dependency-tree adjacency as packed CSR and distance-to-trigger.
// Bit-exact against graph.py:66-75 and data_utils.py:302-323 (on trees/forests).
#include "edg_common.cuh"

namespace edg {

constexpr int kMaxSentence = 4096;
constexpr int kUnreachablePlusOne = 100001;   // data_utils.py:311 + the final "+1" of :323

// head of token i of a sentence whose raw heads start at `hs`.  Malformed heads (out of range, self) are treated as
// roots; of a mutual pair h[i] = j, h[j] = i the higher token becomes a root, so the edge is stored ONCE -- the set
// semantics of graph.py:73-74 (`m[s][t] = m[t][s] = 1`), and what keeps count and fill kernels consistent.
__device__ __forceinline__ int clean_head(const int32_t* __restrict__ hs, int i, int n) {
  const int h = hs[i];
  if (h < 0 || h >= n || h == i) return -1;
  return (hs[h] == i && i > h) ? -1 : h;
}

// ---- extra undirected edges (heads + edges -> CSR) ---------------------------
// Pair e of the edge list belongs to the sentence b with edge_ptr[b] <= e < edge_ptr[b+1] (empty sentences allowed).
__device__ __forceinline__ int pair_sentence(const int32_t* __restrict__ edge_ptr, int B, int e) {
  int lo = 0, hi = B - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (edge_ptr[mid] <= e) lo = mid; else hi = mid - 1;
  }
  return lo;
}

// Pair e as sentence-local (i, j) of the sentence starting at global row `base`.  False for a pair that adds nothing to
// the forest's pattern: an endpoint outside [0, n), i == j, or the edge of a (cleaned) head in either direction.  The
// pair count and scatter passes both decide with this one function, so they agree; duplicates are removed per row by
// extra_sort_kernel.
__device__ __forceinline__ bool extra_pair(const int32_t* __restrict__ heads, const int32_t* __restrict__ sent_ptr,
                                           const int32_t* __restrict__ edges, const int32_t* __restrict__ edge_ptr,
                                           int B, int e, int& base, int& i, int& j) {
  const int b = pair_sentence(edge_ptr, B, e);
  base = sent_ptr[b];
  const int n = sent_ptr[b + 1] - base;
  i = edges[2 * (int64_t)e];
  j = edges[2 * (int64_t)e + 1];
  if (i < 0 || i >= n || j < 0 || j >= n || i == j) return false;
  return clean_head(heads + base, i, n) != j && clean_head(heads + base, j, n) != i;
}

// per-row count of extra entries (both directions of every kept pair); cnt[N] zeroed by the caller
__global__ void pairs_count_kernel(const int32_t* __restrict__ heads, const int32_t* __restrict__ sent_ptr,
                                   const int32_t* __restrict__ edges, const int32_t* __restrict__ edge_ptr, int B, int E,
                                   int32_t* __restrict__ cnt) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  int base, i, j;
  if (e >= E || !extra_pair(heads, sent_ptr, edges, edge_ptr, B, e, base, i, j)) return;
  atomicAdd(&cnt[base + i], 1);
  atomicAdd(&cnt[base + j], 1);
}

// row r's extra neighbours (sentence-local, unordered, maybe repeated) into xl[xoff[r] ..); cur[N] zeroed by the caller
__global__ void pairs_scatter_kernel(const int32_t* __restrict__ heads, const int32_t* __restrict__ sent_ptr,
                                     const int32_t* __restrict__ edges, const int32_t* __restrict__ edge_ptr, int B,
                                     int E, const int32_t* __restrict__ xoff, int32_t* __restrict__ cur,
                                     int32_t* __restrict__ xl) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  int base, i, j;
  if (e >= E || !extra_pair(heads, sent_ptr, edges, edge_ptr, B, e, base, i, j)) return;
  xl[xoff[base + i] + atomicAdd(&cur[base + i], 1)] = j;
  xl[xoff[base + j] + atomicAdd(&cur[base + j], 1)] = i;
}

// One warp per row: sort and de-duplicate the row's extra list in place through a bitmap of the sentence's tokens
// (`words` 32-bit words per warp in shared memory), so the result is a set in ascending order whatever the order of the
// pairs or of the scatter's atomics.  xu[r]: on entry the list length, on return the number of distinct entries.
__global__ void extra_sort_kernel(const int32_t* __restrict__ xoff, int32_t* __restrict__ xl, int32_t* __restrict__ xu,
                                  int N, int words) {
  extern __shared__ uint32_t bm_all[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int r = blockIdx.x * (blockDim.x >> 5) + warp;
  if (r >= N) return;                      // warp-uniform
  const int beg = xoff[r], k = xoff[r + 1] - beg;
  if (k <= 1) return;                      // xu[r] = k already
  uint32_t* bm = bm_all + warp * words;
  for (int q = lane; q < words; q += 32) bm[q] = 0u;
  __syncwarp();
  for (int e = lane; e < k; e += 32) {
    const int c = xl[beg + e];
    if (c >= 32 * words) __trap();         // a sentence longer than the caller's max_len (see heads_fill_kernel)
    atomicOr(&bm[c >> 5], 1u << (c & 31));
  }
  __syncwarp();
  int w = beg;
  for (int q0 = 0; q0 < words; q0 += 32) {
    const int q = q0 + lane;
    uint32_t m = q < words ? bm[q] : 0u;
    const int c = __popc(m);
    int incl = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += t;
    }
    for (int p = w + incl - c; m; m &= m - 1u) xl[p++] = 32 * q + __ffs(m) - 1;
    w += __shfl_sync(0xffffffffu, incl, 31);
  }
  if (lane == 0) xu[r] = w - beg;
}

// ---- heads -> CSR ----------------------------------------------------------
// pass 1: non-zeros of each sentence = n + 2 * (tokens that have a head) [+ the rows' distinct extra entries xu].
// With extras, a sentence over a positive caller bound *nnz_cap fails loudly, and mx[0] collects the largest count.
template <bool kExtra>
__global__ void heads_count_kernel(const int32_t* __restrict__ heads, const int32_t* __restrict__ sent_ptr,
                                   int B, int32_t* __restrict__ sent_nnz, const int32_t* __restrict__ xu = nullptr,
                                   const int32_t* __restrict__ nnz_cap = nullptr, int32_t* __restrict__ mx = nullptr) {
  int b = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (b >= B) return;
  int lane = threadIdx.x & 31;
  int base = sent_ptr[b], n = sent_ptr[b + 1] - base;
  int cnt = 0;
  for (int i = lane; i < n; i += 32) cnt += 1 + 2 * (clean_head(heads + base, i, n) >= 0) + (kExtra ? xu[base + i] : 0);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
  if (lane == 0) {
    sent_nnz[b] = cnt;
    if (kExtra) {
      const int cap = *nnz_cap;
      if (cap > 0 && cnt > cap) __trap();   // the caller's max_sent_nnz is smaller than this sentence: fail loudly
      atomicMax(mx, cnt);
    }
  }
}

// single-block exclusive scan: out[0..n] (n+1 entries), out[n] = total
__global__ void scan_exclusive_kernel(const int32_t* in, int32_t* out, int n) {   // in may alias out
  __shared__ int warp_tot[32];
  __shared__ int carry_s;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5, nw = blockDim.x >> 5;
  if (tid == 0) carry_s = 0;
  __syncthreads();
  for (int base = 0; base < n; base += blockDim.x) {
    int i = base + tid;
    int v = (i < n) ? in[i] : 0;
    int incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      int t = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += t;
    }
    if (lane == 31) warp_tot[wid] = incl;
    __syncthreads();
    if (wid == 0) {
      int w = (lane < nw) ? warp_tot[lane] : 0;
      int wi = w;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        int t = __shfl_up_sync(0xffffffffu, wi, o);
        if (lane >= o) wi += t;
      }
      warp_tot[lane] = wi - w;   // exclusive prefix of the warp totals
    }
    __syncthreads();
    int carry = carry_s;
    if (i < n) out[i] = carry + warp_tot[wid] + incl - v;
    __syncthreads();
    if (tid == blockDim.x - 1) carry_s = carry + warp_tot[wid] + incl;
    __syncthreads();
  }
  if (tid == 0) out[n] = carry_s;
}

// pass 2: one block per sentence; thread i builds row i by scanning the sentence
// in ascending token order, which yields the ascending column order directly.
// With extras, row r's distinct extra neighbours xl[xoff[r] .. + xu[r]) are ascending and disjoint from self, parent
// and children (extra_pair, extra_sort_kernel), so the same scan merges them in; block 0 publishes mx[0].
template <bool kExtra>
__global__ void heads_fill_kernel(const int32_t* __restrict__ heads, const int32_t* __restrict__ sent_ptr,
                                  const int32_t* __restrict__ sent_off, int32_t* __restrict__ row_ptr,
                                  int32_t* __restrict__ col, int32_t* __restrict__ row_sent, int B, int N, int cap,
                                  const int32_t* __restrict__ xoff = nullptr, const int32_t* __restrict__ xl = nullptr,
                                  const int32_t* __restrict__ xu = nullptr, const int32_t* __restrict__ mx = nullptr,
                                  int32_t* __restrict__ sent_max_nnz = nullptr) {
  extern __shared__ int32_t sm[];
  const int b = blockIdx.x;
  const int base = sent_ptr[b], n = sent_ptr[b + 1] - base;
  if (n > cap) __trap();      // the caller's max_len (it sizes the shared arrays) is smaller than this sentence: fail loudly
  if (kExtra && b == 0 && threadIdx.x == 0) *sent_max_nnz = *mx;
  int32_t* h = sm;            // cleaned heads [n]
  int32_t* deg = sm + n;      // row lengths -> exclusive offsets [n+1]
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    h[i] = clean_head(heads + base, i, n);
    deg[i] = 0;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    atomicAdd(&deg[i], 1 + (h[i] >= 0) + (kExtra ? xu[base + i] : 0));
    if (h[i] >= 0) atomicAdd(&deg[h[i]], 1);
  }
  __syncthreads();
  if (threadIdx.x < 32) {     // warp scan over the sentence (n <= 4096)
    int lane = threadIdx.x, carry = 0;
    for (int s = 0; s < n; s += 32) {
      int i = s + lane;
      int v = (i < n) ? deg[i] : 0, incl = v;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        int t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
      }
      if (i < n) deg[i] = carry + incl - v;
      carry += __shfl_sync(0xffffffffu, incl, 31);
    }
    if (lane == 0) deg[n] = carry;
  }
  __syncthreads();
  const int off0 = sent_off[b];
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    int w = off0 + deg[i];
    row_ptr[base + i] = w;
    row_sent[base + i] = b;
    const int hi = h[i];
    if (kExtra) {
      int xp = xoff[base + i];
      const int xe = xp + xu[base + i];
      for (int k = 0; k < n; ++k) {
        bool nz = k == i || k == hi || h[k] == i;
        if (!nz && xp < xe && xl[xp] == k) { nz = true; ++xp; }
        if (nz) col[w++] = base + k;
      }
    } else {
      for (int k = 0; k < n; ++k)
        if (k == i || k == hi || h[k] == i) col[w++] = base + k;
    }
  }
  if (b == B - 1 && threadIdx.x == 0) row_ptr[N] = off0 + deg[n];
}

// ---- dense [B,T,T] -> CSR ----------------------------------------------------
template <typename T>
__global__ void dense_count_kernel(const T* __restrict__ adj, int rows, int Tn, int64_t sb, int64_t sr,
                                   int64_t sc, int32_t* __restrict__ deg, int32_t* __restrict__ flags) {
  int r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (r >= rows) return;
  int lane = threadIdx.x & 31;
  int b = r / Tn, i = r - b * Tn;
  const T* row = adj + b * sb + i * sr;
  int cnt = 0, odd = 0, asym = 0;
  for (int j = lane; j < Tn; j += 32) {
    T v = row[j * sc];
    if (v != T(0)) {
      ++cnt;
      if (v != T(1)) ++odd;
      if (adj[b * sb + j * sr + i * sc] == T(0)) ++asym;
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    odd += __shfl_xor_sync(0xffffffffu, odd, o);
    asym += __shfl_xor_sync(0xffffffffu, asym, o);
  }
  if (lane == 0) {
    deg[r] = cnt;
    if (odd) atomicAdd(&flags[0], odd);
    if (asym) atomicAdd(&flags[1], asym);
  }
}

template <typename T>
__global__ void dense_fill_kernel(const T* __restrict__ adj, int rows, int Tn, int64_t sb, int64_t sr,
                                  int64_t sc, const int32_t* __restrict__ row_ptr, int32_t* __restrict__ col) {
  int r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (r >= rows) return;
  int lane = threadIdx.x & 31;
  int b = r / Tn, i = r - b * Tn;
  const T* row = adj + b * sb + i * sr;
  int w = row_ptr[r];
  for (int j0 = 0; j0 < Tn; j0 += 32) {
    int j = j0 + lane;
    bool nz = (j < Tn) && (row[j * sc] != T(0));
    unsigned m = __ballot_sync(0xffffffffu, nz);
    if (nz) col[w + __popc(m & ((1u << lane) - 1u))] = b * Tn + j;
    w += __popc(m);
  }
}

// ---- distance to the trigger -------------------------------------------------
// one block per sentence, level-synchronous BFS over the CSR (true hop counts;
// equals data_utils.py:302-323 on trees and forests, SURVEY fact 8).
// level-synchronous BFS of one sentence (rows base .. base + n - 1) from sentence-local row `a`, written to out[0..n)
__device__ __forceinline__ void bfs_sentence(const int32_t* __restrict__ row_ptr, const int32_t* __restrict__ col, int base,
                                             int n, int a, int32_t* __restrict__ out, int32_t* d) {
  for (int i = threadIdx.x; i < n; i += blockDim.x) d[i] = -1;
  __syncthreads();
  if (threadIdx.x == 0 && a >= 0 && a < n) d[a] = 0;
  __syncthreads();
  for (int level = 0; level < n; ++level) {
    int grew = 0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
      if (d[i] == level) {
        for (int e = row_ptr[base + i]; e < row_ptr[base + i + 1]; ++e) {
          int j = col[e] - base;
          if (d[j] < 0) { d[j] = level + 1; grew = 1; }   // same value from every writer
        }
      }
    }
    if (!__syncthreads_or(grew)) break;
  }
  for (int i = threadIdx.x; i < n; i += blockDim.x)
    out[i] = d[i] >= 0 ? d[i] + 1 : kUnreachablePlusOne;
}

// one block per sentence, level-synchronous BFS over the CSR (true hop counts;
// equals data_utils.py:302-323 on trees and forests, SURVEY fact 8).
__global__ void tree_dist_kernel(const int32_t* __restrict__ row_ptr, const int32_t* __restrict__ col,
                                 const int32_t* __restrict__ sent_ptr, const int32_t* __restrict__ anchor,
                                 int32_t* __restrict__ dist, int cap) {
  extern __shared__ int32_t d[];
  const int b = blockIdx.x;
  const int base = sent_ptr[b], n = sent_ptr[b + 1] - base;
  if (n > cap) __trap();      // max_len smaller than this sentence (see heads_fill_kernel)
  bfs_sentence(row_ptr, col, base, n, anchor[b], dist + base, d);
}

// the same per (sentence, trigger) pair: block p walks sentence pair_sent[p] from anchor[p] and writes that pair's copy
// of the sentence's distances at pair_row_ptr[p]
__global__ void tree_dist_pairs_kernel(const int32_t* __restrict__ row_ptr, const int32_t* __restrict__ col,
                                       const int32_t* __restrict__ sent_ptr, const int32_t* __restrict__ pair_sent,
                                       const int32_t* __restrict__ pair_row_ptr, const int32_t* __restrict__ anchor,
                                       int32_t* __restrict__ dist, int cap) {
  extern __shared__ int32_t d[];
  const int p = blockIdx.x;
  const int s = pair_sent[p];
  const int base = sent_ptr[s], n = sent_ptr[s + 1] - base;
  if (n > cap) __trap();      // max_len smaller than this sentence
  bfs_sentence(row_ptr, col, base, n, anchor[p], dist + pair_row_ptr[p], d);
}

__global__ void dist_pad_kernel(const int32_t* __restrict__ dist, const int32_t* __restrict__ sent_ptr,
                                int Tn, int pad_mode, int64_t* __restrict__ out) {
  const int b = blockIdx.x;
  const int base = sent_ptr[b], n = min(sent_ptr[b + 1] - base, Tn);
  __shared__ int fill_s;
  if (threadIdx.x < 32) {
    int m = 0;
    for (int i = threadIdx.x; i < n; i += 32) m = max(m, dist[base + i]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
    if (threadIdx.x == 0) fill_s = (pad_mode == EDG_PAD_ZERO) ? 0 : m + 1;
  }
  __syncthreads();
  const int fill = fill_s;
  for (int t = threadIdx.x; t < Tn; t += blockDim.x)
    out[(int64_t)b * Tn + t] = (t < n) ? dist[base + t] : fill;
}

}  // namespace edg

using namespace edg;

extern "C" int edg_csr_from_heads(const int32_t* heads, const int32_t* sent_ptr, int32_t B, int32_t N,
                                  int32_t max_len, int32_t* row_ptr, int32_t* col, int32_t* row_sent,
                                  int32_t* ws, edg_stream stream) {
  if (B < 0 || N < 0) return EDG_ERR_ARG;
  if (!sent_ptr || !row_ptr || !ws) return EDG_ERR_ARG;
  if (N > 0 && (!heads || !col || !row_sent)) return EDG_ERR_ARG;
  if (max_len > kMaxSentence) return EDG_ERR_UNSUPPORTED;
  cudaStream_t s = (cudaStream_t)stream;
  if (B == 0) { cudaMemsetAsync(row_ptr, 0, sizeof(int32_t), s); return check_launch(); }
  int32_t* sent_nnz = ws;   // B ints, scanned in place into B+1 offsets
  heads_count_kernel<false><<<(B + 7) / 8, 256, 0, s>>>(heads, sent_ptr, B, sent_nnz);
  scan_exclusive_kernel<<<1, 1024, 0, s>>>(sent_nnz, sent_nnz, B);
  int threads = max_len <= 64 ? 64 : (max_len <= 128 ? 128 : 256);
  size_t smem = (2 * (size_t)max_len + 1) * sizeof(int32_t);
  heads_fill_kernel<false><<<B, threads, smem, s>>>(heads, sent_ptr, sent_nnz, row_ptr, col, row_sent, B, N, max_len);
  return check_launch();
}

// workspace of edg_csr_from_heads_edges, in int32: sentence counts -> offsets [B+1] | extra entries per row -> offsets
// [N+1] | distinct extra entries per row [N] | largest sentence count [1] | extra lists [2E]
static size_t heads_edges_ws_ints(int64_t B, int64_t N, int64_t E) { return (B + 1) + (N + 1) + N + 1 + 2 * E; }

extern "C" size_t edg_csr_from_heads_edges_workspace(int32_t B, int32_t N, int32_t E) {
  if (B < 0 || N < 0 || E < 0) return 0;
  return heads_edges_ws_ints(B, N, E) * sizeof(int32_t);
}

extern "C" int edg_csr_from_heads_edges(const int32_t* heads, const int32_t* sent_ptr, const int32_t* edges,
                                        const int32_t* edge_ptr, int32_t B, int32_t N, int32_t E, int32_t max_len,
                                        int32_t* row_ptr, int32_t* col, int32_t* row_sent, int32_t* sent_max_nnz,
                                        void* ws, size_t ws_bytes, edg_stream stream) {
  if (B < 0 || N < 0 || E < 0 || max_len < 0) return EDG_ERR_ARG;
  if (!sent_ptr || !row_ptr || !sent_max_nnz || !ws) return EDG_ERR_ARG;
  if (N > 0 && (!heads || !col || !row_sent)) return EDG_ERR_ARG;
  if (E > 0 && (!edges || !edge_ptr)) return EDG_ERR_ARG;
  if (max_len > kMaxSentence) return EDG_ERR_UNSUPPORTED;
  if (ws_bytes < edg_csr_from_heads_edges_workspace(B, N, E)) return EDG_ERR_WORKSPACE;
  cudaStream_t s = (cudaStream_t)stream;
  if (B == 0) {
    cudaMemsetAsync(row_ptr, 0, sizeof(int32_t), s);
    cudaMemsetAsync(sent_max_nnz, 0, sizeof(int32_t), s);
    return check_launch();
  }
  int32_t* sent_nnz = (int32_t*)ws;
  int32_t* xoff = sent_nnz + (B + 1);
  int32_t* xu = xoff + (N + 1);
  int32_t* mx = xu + N;
  int32_t* xl = mx + 1;
  cudaMemsetAsync(xoff, 0, (2 * (size_t)N + 2) * sizeof(int32_t), s);     // xoff, xu, mx
  if (E > 0 && N > 0) {
    const int words = max(1, (max_len + 31) / 32);
    pairs_count_kernel<<<(E + 255) / 256, 256, 0, s>>>(heads, sent_ptr, edges, edge_ptr, B, E, xoff);
    scan_exclusive_kernel<<<1, 1024, 0, s>>>(xoff, xoff, N);
    pairs_scatter_kernel<<<(E + 255) / 256, 256, 0, s>>>(heads, sent_ptr, edges, edge_ptr, B, E, xoff, xu, xl);
    extra_sort_kernel<<<(N + 7) / 8, 256, 8 * words * sizeof(uint32_t), s>>>(xoff, xl, xu, N, words);
  }
  heads_count_kernel<true><<<(B + 7) / 8, 256, 0, s>>>(heads, sent_ptr, B, sent_nnz, xu, sent_max_nnz, mx);
  scan_exclusive_kernel<<<1, 1024, 0, s>>>(sent_nnz, sent_nnz, B);
  int threads = max_len <= 64 ? 64 : (max_len <= 128 ? 128 : 256);
  size_t smem = (2 * (size_t)max_len + 1) * sizeof(int32_t);
  heads_fill_kernel<true><<<B, threads, smem, s>>>(heads, sent_ptr, sent_nnz, row_ptr, col, row_sent, B, N, max_len,
                                                   xoff, xl, xu, mx, sent_max_nnz);
  return check_launch();
}

extern "C" int edg_csr_from_dense_count(const void* adj, int adj_is_i64, int32_t B, int32_t T,
                                        int64_t stride_b, int64_t stride_r, int64_t stride_c,
                                        int32_t* row_ptr, int32_t* flags, edg_stream stream) {
  if (!adj || !row_ptr || !flags || B <= 0 || T <= 0) return EDG_ERR_ARG;
  if ((int64_t)B * T > (1ll << 30)) return EDG_ERR_UNSUPPORTED;
  cudaStream_t s = (cudaStream_t)stream;
  int rows = B * T;
  cudaMemsetAsync(flags, 0, 2 * sizeof(int32_t), s);
  int blocks = (rows + 7) / 8;
  if (adj_is_i64)
    dense_count_kernel<long long><<<blocks, 256, 0, s>>>((const long long*)adj, rows, T, stride_b, stride_r, stride_c, row_ptr, flags);
  else
    dense_count_kernel<float><<<blocks, 256, 0, s>>>((const float*)adj, rows, T, stride_b, stride_r, stride_c, row_ptr, flags);
  scan_exclusive_kernel<<<1, 1024, 0, s>>>(row_ptr, row_ptr, rows);
  return check_launch();
}

extern "C" int edg_csr_from_dense_fill(const void* adj, int adj_is_i64, int32_t B, int32_t T,
                                       int64_t stride_b, int64_t stride_r, int64_t stride_c,
                                       const int32_t* row_ptr, int32_t* col, edg_stream stream) {
  if (!adj || !row_ptr || !col || B <= 0 || T <= 0) return EDG_ERR_ARG;
  cudaStream_t s = (cudaStream_t)stream;
  int rows = B * T;
  int blocks = (rows + 7) / 8;
  if (adj_is_i64)
    dense_fill_kernel<long long><<<blocks, 256, 0, s>>>((const long long*)adj, rows, T, stride_b, stride_r, stride_c, row_ptr, col);
  else
    dense_fill_kernel<float><<<blocks, 256, 0, s>>>((const float*)adj, rows, T, stride_b, stride_r, stride_c, row_ptr, col);
  return check_launch();
}

extern "C" int edg_tree_dist(const int32_t* row_ptr, const int32_t* col, const int32_t* sent_ptr,
                             const int32_t* anchor, int32_t B, int32_t max_len, int32_t* dist,
                             edg_stream stream) {
  if (B < 0) return EDG_ERR_ARG;
  if (B == 0) return EDG_OK;
  if (!row_ptr || !col || !sent_ptr || !anchor || !dist) return EDG_ERR_ARG;
  if (max_len > 8192) return EDG_ERR_UNSUPPORTED;
  int threads = max_len <= 64 ? 64 : (max_len <= 128 ? 128 : 256);
  tree_dist_kernel<<<B, threads, (size_t)max_len * sizeof(int32_t), (cudaStream_t)stream>>>(row_ptr, col, sent_ptr, anchor, dist, max_len);
  return check_launch();
}

extern "C" int edg_tree_dist_pairs(const int32_t* row_ptr, const int32_t* col, const int32_t* sent_ptr,
                                   const int32_t* pair_sent, const int32_t* pair_row_ptr, const int32_t* anchor, int32_t P,
                                   int32_t max_len, int32_t* dist, edg_stream stream) {
  if (P < 0 || max_len < 0) return EDG_ERR_ARG;
  if (P == 0) return EDG_OK;
  if (!row_ptr || !col || !sent_ptr || !pair_sent || !pair_row_ptr || !anchor || !dist) return EDG_ERR_ARG;
  if (max_len > 8192) return EDG_ERR_UNSUPPORTED;
  int threads = max_len <= 64 ? 64 : (max_len <= 128 ? 128 : 256);
  tree_dist_pairs_kernel<<<P, threads, (size_t)(max_len > 0 ? max_len : 1) * sizeof(int32_t), (cudaStream_t)stream>>>(
      row_ptr, col, sent_ptr, pair_sent, pair_row_ptr, anchor, dist, max_len);
  return check_launch();
}

extern "C" int edg_dist_pad(const int32_t* dist, const int32_t* sent_ptr, int32_t B, int32_t T,
                            int pad_mode, int64_t* out, edg_stream stream) {
  if (B < 0 || T <= 0) return EDG_ERR_ARG;
  if (B == 0) return EDG_OK;
  if (!dist || !sent_ptr || !out) return EDG_ERR_ARG;
  if (pad_mode != EDG_PAD_MAX_PLUS_1 && pad_mode != EDG_PAD_ZERO) return EDG_ERR_ARG;
  dist_pad_kernel<<<B, 128, 0, (cudaStream_t)stream>>>(dist, sent_ptr, T, pad_mode, out);
  return check_launch();
}
