// gcn_layer : one graph-convolution layer (models/gcn.py:33-45) as ONE kernel, projection first:
//
//     forward   y = A^ (x W) + b          A^ = D^-1 A  (A = tree adjacency with self loops, deg = rowsum(A),
//     adjoint   y = A^T ((x W) + patch)                 D = diag(deg + 1): `adj @ hidden / (rowsum + 1)`)
//
// which is the association the reference itself uses (`torch.matmul(adj, torch.matmul(text, W)) / denom + b`).
// Both directions of a training step have this shape: with u_l = h_{l-1} W_l and h_l = A^ u_l + b_l the backward
// pass is  du_l = A^T dh_l,  dW_l = h_{l-1}^T du_l,  dh_{l-1} = du_l W_l^T  -- so the kernel that produces
// dh_{l-1} = du_l W_l^T also applies the NEXT adjoint aggregation in its epilogue and writes du_{l-1}; the
// aggregated rows never exist in HBM in either direction.
//
// A tile = a run of WHOLE sentences with at most `rows_cap` (<= 128) token rows (edg_tile_plan), so every
// neighbour of a tile row is a tile row and the max-pool over a sentence's tokens completes inside the tile.
//   warp 0      TMA producer: the tile's rows as [32 x 64] SW128 boxes into a K-block ring (only the 32-row
//               boxes that hold rows are fetched); once, the CTA's weight slice (stationary for its whole life)
//   warp 1      single-thread tcgen05.mma issuer, M = 128, N = the CTA's column slice (<= 160), 3 TMEM stages
//   warp 2      stages the NEXT tiles' CSR slice (tile-local u8 neighbour ids, u16 row offsets) in shared memory
//   warps 4..   epilogue, per column pass:
//               A  tcgen05.ld -> (adjoint: x 1/(deg+1)) -> fp32 staging tile in shared memory (XOR-swizzled 16-byte
//                  chunks: conflict-free for the row-per-lane stores here and the chunk-per-lane loads of B)
//               P  (adjoint, optional) patch: staging[arg[s,c]][c] += val[s,c]  -- the gradient the gated max-pool
//                  views of layer 1 route to their arg-max rows (bert_amir5.py:627-638)
//               B  thread = (16-byte column chunk, row slice): y_i = sum_{j in row i} S_j (x 1/(deg_i+1) + bias
//                  forward) -> bf16, a warp writes 256+ contiguous bytes of a row;  forward: running max of
//                  (ordered bf16 value << 16 | 0xffff - row) keys per sentence -> shared-memory atomicMax -> the
//                  column maximum and its FIRST row (torch.max semantics) for the gated max-pools;  adjoint:
//                  column sums of the un-aggregated rows (the bias gradient) ride along in registers
// N is split over two CTAs when it exceeds 160 columns (D = 300: 160 + 144); the two CTAs of a tile run side by
// side, so the second read of the tile's rows is an L2 hit.
//
// Unity build: included after edg_gemm_tc.cu (PTX wrappers, descriptors, TMA map helper).
#include <stdlib.h>

#include "edg_common.cuh"

namespace edg {

constexpr int kFRows = 128;             // UMMA M
constexpr int kFMaxSent = 6;            // sentences per tile (pool table rows)
constexpr int kFMaxNnz = 512;           // CSR entries per tile (a tree of n rows has 3n - 2)
constexpr int kFAccStages = 3;
constexpr int kFAccStride = 160;        // TMEM columns per accumulator stage
constexpr int kFMaxStages = 6;          // K-block ring
constexpr int kFCsrBufs = 3;
constexpr int kFCsrBytes = 32 + 16 * 128;  // per buffer: hdr 16 | sent_first u8[16] | row words uint4[128]
constexpr int kFScratch = 272 + 512;    // per stager warp: rp u16[136] | col u8[512] (raw CSR slice of the tile being staged)
constexpr int kFLut = 136;              // 1/(d+1) for d < 136
constexpr int kFMaxEpiWarps = 12;

struct GcnLayerParams {
  CUtensorMap map_a;                    // [N, K] bf16 rows, box [32 rows x 64 cols], SW128
  CUtensorMap map_w;                    // [Nout, K] bf16 (row n = weights of output column n), box [16 x 64], SW128
  const int32_t* tile_info;             // [n_tiles][8] = s0, s1, r0, r1, e0, e1, -, -
  const int32_t* n_tiles;               // device scalar
  const int32_t* row_ptr;
  const int32_t* col;
  const int32_t* sent_ptr;
  const float* bias;                    // [Nout] or null (forward)
  __nv_bfloat16* y;
  int64_t ldy;
  float* hmax;                          // [B, ldpool] column maxima or null (forward)
  int32_t* harg;                        // [B, ldpool] global row of the maximum (-1: empty sentence)
  int64_t ldpool;
  const float* patch_val;               // [B, ldpatch] or null (adjoint)
  const int32_t* patch_arg;             // [B, ldpatch] global row, < 0 = none
  int64_t ldpatch;
  float* colsum_part;                   // [gridDim.x / n_split][Nout] partial column sums or null (adjoint)
  long long* trace;                     // bring-up only (EDG_FUSED_DEBUG & 32): clock64 timeline of CTA 0's epilogue
  int K, Nout, num_kb, mode, n_split, npass, stages, rows_cap, debug;
  int bn[2];                            // columns of CTA half 0 / 1 (multiples of 16)
  uint32_t idesc[2];
  int pitch;                            // staging row pitch in bytes: columns * 2 + 16 (bf16; an odd number of 16-byte chunks, so the
                                        // row-per-lane stores of phase A and the chunk-per-lane loads of phase B are conflict-free)
  int box_rows;                         // rows per TMA box of the activation tile (32, 64 or 128)
  int sleep_ns;                         // back-off of the helper warps' long waits
  int prefetch;                         // tiles of look-ahead for the TMA L2 prefetch (0 = off)
  uint32_t off_a, off_s, off_tab, off_csr, off_scr, off_lut, off_bar;   // shared-memory offsets (W at 0)
};

__device__ __forceinline__ void tmem_ld_32x32_x16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
}
__device__ __forceinline__ void lds_v4(uint32_t addr, float (&v)[4]) {
  uint32_t a, b, c, d;
  asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(a), "=r"(b), "=r"(c), "=r"(d) : "r"(addr));
  v[0] = __uint_as_float(a); v[1] = __uint_as_float(b); v[2] = __uint_as_float(c); v[3] = __uint_as_float(d);
}
__device__ __forceinline__ void epi_bar(int nthreads) { asm volatile("bar.sync 1, %0;" ::"r"(nthreads) : "memory"); }

// wait on an mbarrier phase; the hardware may park the thread for up to `hint_ns` per attempt (it wakes on completion),
// so a waiting warp costs a few instructions per microsecond instead of a tight polling loop
__device__ __forceinline__ void f2_wait(uint32_t bar, uint32_t parity, uint32_t hint_ns = 1000) {
  uint32_t ok = 0, spins = 0;
  while (true) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok) : "r"(bar), "r"(parity), "r"(hint_ns) : "memory");
    if (ok) break;
    if (++spins > (1u << 20)) __trap();
  }
}

// (the helper warps' long waits used to poll with __nanosleep back-off: 20 % of the kernel's executed instructions were
// polling loops competing with the epilogue warps of the same scheduler)
__device__ __forceinline__ void mbar_wait_relaxed(uint32_t bar, uint32_t parity, uint32_t = 0) { f2_wait(bar, parity); }

// order-preserving key of a bf16 value held in the UPPER 16 bits of x (lower 16 ignored) | low field
__device__ __forceinline__ uint32_t pool_key(uint32_t x, uint32_t low) {
  const uint32_t m = (uint32_t)((int32_t)x >> 31) | 0x80000000u;
  return ((x ^ m) & 0xffff0000u) | low;
}
__device__ __forceinline__ float pool_key_value(uint32_t key) {
  const uint32_t o = key & 0xffff0000u;
  return __uint_as_float((o & 0x80000000u) ? (o ^ 0x80000000u) : (~o & 0xffff0000u));
}

template <int EPI_WARPS>
__global__ void __launch_bounds__((4 + EPI_WARPS) * 32, 1)
gcn_layer_kernel(const __grid_constant__ GcnLayerParams P) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  constexpr int kEpiThreads = EPI_WARPS * 32;
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* sm = smem_raw + (base - smem_u32(smem_raw));
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int half = (P.n_split == 2) ? (int)(blockIdx.x & 1) : 0;
  const int t_first = (P.debug & 64) ? (int)blockIdx.x : (int)blockIdx.x / P.n_split;      // bit 64 (bring-up): one tile per CTA, timing only
  const int t_step = (P.debug & 64) ? (int)gridDim.x : (int)gridDim.x / P.n_split;
  const int n0 = half * P.bn[0];
  const int bn = P.bn[half];
  const int num_kb = P.num_kb;
  const uint32_t w_kb_bytes = (uint32_t)bn * 128u;
  auto Wblk = [&](int kb) { return base + (uint32_t)kb * w_kb_bytes; };
  auto Ablk = [&](int s) { return base + P.off_a + (uint32_t)s * 16384u; };
  const uint32_t bars = base + P.off_bar;
  auto full = [&](int s) { return bars + 8 * s; };
  auto empty = [&](int s) { return bars + 8 * (kFMaxStages + s); };
  auto tfull = [&](int s) { return bars + 8 * (2 * kFMaxStages + s); };
  auto tempty = [&](int s) { return bars + 8 * (2 * kFMaxStages + kFAccStages + s); };
  auto cfull = [&](int s) { return bars + 8 * (2 * kFMaxStages + 2 * kFAccStages + s); };
  auto cempty = [&](int s) { return bars + 8 * (2 * kFMaxStages + 2 * kFAccStages + kFCsrBufs + s); };
  const uint32_t wfull = bars + 8 * (2 * kFMaxStages + 2 * kFAccStages + 2 * kFCsrBufs);
  const uint32_t tmem_slot = wfull + 8;
  const uint32_t lut_s = base + P.off_lut;
  float* lut = reinterpret_cast<float*>(sm + P.off_lut);

  for (int i = threadIdx.x; i < kFLut; i += blockDim.x) lut[i] = __frcp_rn((float)(i + 1));
  if (threadIdx.x == 0) {
    tma_prefetch_desc(&P.map_a);
    tma_prefetch_desc(&P.map_w);
    for (int s = 0; s < P.stages; ++s) { mbar_init(full(s), 1); mbar_init(empty(s), 1); }
    for (int s = 0; s < kFAccStages; ++s) { mbar_init(tfull(s), 1); mbar_init(tempty(s), EPI_WARPS); }
    for (int s = 0; s < kFCsrBufs; ++s) { mbar_init(cfull(s), 1); mbar_init(cempty(s), EPI_WARPS); }
    mbar_init(wfull, 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));
  const int n_tiles = __ldg(P.n_tiles);

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer
    if (lane == 0) {
      mbar_expect_tx(wfull, (uint32_t)num_kb * w_kb_bytes);
      for (int kb = 0; kb < num_kb; ++kb)
        for (int r = 0; r < bn; r += 16) tma_load_2d(Wblk(kb) + (uint32_t)r * 128u, &P.map_w, wfull, kb * 64, n0 + r);
      int stage = 0; uint32_t phase = 0;
      // row ranges of this CTA's next tiles, kept kPfDepth + 1 tiles ahead so that neither the loads nor the L2
      // prefetches ever wait for a tile_info load issued in the same iteration
      constexpr int kAhead = 4;
      int rr0[kAhead], rr1[kAhead];
#pragma unroll
      for (int a = 0; a < kAhead; ++a) {
        const int ta = t_first + a * t_step;
        rr0[a] = 0; rr1[a] = 0;
        if (ta < n_tiles) { rr0[a] = __ldg(P.tile_info + 8 * ta + 2); rr1[a] = __ldg(P.tile_info + 8 * ta + 3); }
      }
      const int pf = (half == 0) ? P.prefetch : 0;        // one CTA of the pair prefetches for both
      for (int t = t_first; t < n_tiles; t += t_step) {
        const int r0 = rr0[0], r1 = rr1[0];
        int pr0 = 0, pr1 = 0;
        if (pf == 1) { pr0 = rr0[1]; pr1 = rr1[1]; } else if (pf == 2) { pr0 = rr0[2]; pr1 = rr1[2]; } else if (pf == 3) { pr0 = rr0[3]; pr1 = rr1[3]; }
#pragma unroll
        for (int a = 0; a + 1 < kAhead; ++a) { rr0[a] = rr0[a + 1]; rr1[a] = rr1[a + 1]; }
        const int tn = t + kAhead * t_step;
        rr0[kAhead - 1] = 0; rr1[kAhead - 1] = 0;
        if (tn < n_tiles) { rr0[kAhead - 1] = __ldg(P.tile_info + 8 * tn + 2); rr1[kAhead - 1] = __ldg(P.tile_info + 8 * tn + 3); }
        // the rows of the tile `pf` steps ahead -> L2 (fire and forget): the loads below then see L2 latency
        for (int r = pr0; r < pr1; r += 32)
          for (int kb = 0; kb < num_kb; ++kb)
            asm volatile("cp.async.bulk.prefetch.tensor.2d.L2.global.tile [%0, {%1, %2}];"
                         ::"l"(reinterpret_cast<uint64_t>(&P.map_a)), "r"(kb * 64), "r"(r) : "memory");
        const int nb32 = (P.debug & 8) ? 0 : (r1 - r0 + P.box_rows - 1) / P.box_rows;
        const uint32_t box_bytes = (uint32_t)P.box_rows * 128u;
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait_relaxed(empty(stage), phase ^ 1, (uint32_t)P.sleep_ns);
          mbar_expect_tx(full(stage), (uint32_t)nb32 * box_bytes);
          for (int b = 0; b < nb32; ++b)
            tma_load_2d(Ablk(stage) + (uint32_t)b * box_bytes, &P.map_a, full(stage), kb * 64, r0 + P.box_rows * b);
          if (++stage == P.stages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer
    if (lane == 0) {
      const uint32_t idesc = P.idesc[half];
      f2_wait(wfull, 0);
      int stage = 0; uint32_t phase = 0;
      int it = 0;
      for (int t = t_first; t < n_tiles; t += t_step, ++it) {
        const int as = it % kFAccStages;
        const uint32_t aphase = (uint32_t)(it / kFAccStages) & 1u;
        mbar_wait_relaxed(tempty(as), aphase ^ 1, (uint32_t)P.sleep_ns);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(as * kFAccStride);
        for (int kb = 0; kb < num_kb; ++kb) {
          f2_wait(full(stage), phase);
          tc_fence_after();
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            if (kb * 64 + k * 16 < P.K && !(P.debug & 16)) {
              const uint64_t ad = make_desc_sw128(Ablk(stage) + k * 32, 16, 1024);
              const uint64_t bd = make_desc_sw128(Wblk(kb) + k * 32, 16, 1024);
              umma_bf16(d_tmem, ad, bd, idesc, (kb | k) != 0);
            }
          }
          umma_commit(empty(stage));
          if (++stage == P.stages) { stage = 0; phase ^= 1; }
        }
        umma_commit(tfull(as));
      }
    }
  } else if (warp < 4) {
    // ------------------------------------------------------------------ CSR stagers (warp 2: even tiles, warp 3: odd)
    // per tile: raw CSR slice -> this warp's scratch with batched, coalesced loads (two latency rounds), then one
    // 16-byte word per row: self + the first seven other neighbours as tile-local u8 ids (unused slots = the zero
    // row of the staging tile) | entry count | sentence | first raw CSR entry, so that phase B needs ONE
    // shared-memory load per row before its gathers and no branches for rows with <= 4 entries
    uint16_t* rp = reinterpret_cast<uint16_t*>(sm + P.off_scr + (warp - 2) * kFScratch);
    uint8_t* cl = sm + P.off_scr + (warp - 2) * kFScratch + 272;
    const uint32_t zrow = (uint32_t)P.rows_cap;
    for (int it = warp - 2, t = t_first + (warp - 2) * t_step; t < n_tiles; t += 2 * t_step, it += 2) {
      const int cb = it % kFCsrBufs;
      const uint32_t cphase = (uint32_t)(it / kFCsrBufs) & 1u;
      int v = (lane < 6) ? __ldg(P.tile_info + 8 * t + lane) : 0;      // issued before blocking on the buffer
      const int s0 = __shfl_sync(0xffffffffu, v, 0), s1 = __shfl_sync(0xffffffffu, v, 1);
      const int r0 = __shfl_sync(0xffffffffu, v, 2), r1 = __shfl_sync(0xffffffffu, v, 3);
      const int e0 = __shfl_sync(0xffffffffu, v, 4), e1 = __shfl_sync(0xffffffffu, v, 5);
      const int n = (P.debug & 4) ? 0 : r1 - r0, ns = (P.debug & 4) ? 0 : s1 - s0, nnz = (P.debug & 4) ? 0 : min(e1 - e0, kFMaxNnz);
      int rpv[5], cv[16], sf = 0;
#pragma unroll
      for (int k = 0; k < 5; ++k) { const int i = lane + 32 * k; rpv[k] = (i <= n) ? __ldg(P.row_ptr + r0 + i) : 0; }
#pragma unroll
      for (int k = 0; k < 16; ++k) { const int i = lane + 32 * k; cv[k] = (i < nnz) ? __ldg(P.col + e0 + i) : 0; }
      if (lane <= ns) sf = __ldg(P.sent_ptr + s0 + lane);
#pragma unroll
      for (int k = 0; k < 5; ++k) { const int i = lane + 32 * k; if (i <= n) rp[i] = (uint16_t)(rpv[k] - e0); }
#pragma unroll
      for (int k = 0; k < 16; ++k) { const int i = lane + 32 * k; if (i < nnz) cl[i] = (uint8_t)(cv[k] - r0); }
      mbar_wait_relaxed(cempty(cb), cphase ^ 1, (uint32_t)P.sleep_ns);
      uint8_t* cs = sm + P.off_csr + cb * kFCsrBytes;
      int32_t* hdr = reinterpret_cast<int32_t*>(cs);
      uint8_t* sfirst = cs + 16;
      uint4* meta = reinterpret_cast<uint4*>(cs + 32);
      if (lane <= ns) sfirst[lane] = (uint8_t)(sf - r0);
      __syncwarp();
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int i = lane + 32 * k;
        if (i < n) {
          const int e_beg = rp[i], deg = rp[i + 1] - e_beg;
          uint64_t ids = (zrow * 0x0101010101010101ull & ~0xffull) | (uint64_t)i;
          int cnt = 0;
          for (int q = 0; q < 8 && q < deg; ++q) {
            const uint32_t j = cl[e_beg + q];
            if ((int)j != i && cnt < 7) { ++cnt; ids = (ids & ~(0xffull << (8 * cnt))) | ((uint64_t)j << (8 * cnt)); }
          }
          int s = 0;
          for (int q = 1; q < ns; ++q) s += (sfirst[q] <= i) ? 1 : 0;   // last sentence whose first row is <= i
          meta[i] = make_uint4((uint32_t)ids, (uint32_t)(ids >> 32), (uint32_t)deg | ((uint32_t)s << 8), (uint32_t)(e0 + e_beg));
        }
      }
      if (lane == 0) { hdr[0] = r0; hdr[1] = n; hdr[2] = ns; hdr[3] = s0; }
      __syncwarp();
      if (lane == 0) mbar_arrive(cfull(cb));
    }
  } else {
    // ------------------------------------------------------------------ epilogue
    const int ew = warp - 4;
    const int q = warp & 3;
    const int part = ew >> 2;
    constexpr int nparts = EPI_WARPS / 4;
    const int et = threadIdx.x - 128;                       // 0 .. kEpiThreads-1
    const uint32_t s_base = base + P.off_s;
    uint32_t* tab = reinterpret_cast<uint32_t*>(sm + P.off_tab);
    const int pitch = P.pitch;
    const int cw = bn;                                      // columns of this CTA's slice (multiple of 16)
    const int tabw = P.bn[0];                               // table row pitch
    const bool pool = P.hmax != nullptr;
    const bool patch = P.patch_val != nullptr;
    // phase B mapping: thread = (8-column chunk k8, row slice sl)
    const int nch = cw >> 3;
    const int nsl = kEpiThreads / nch;
    const int sl = et / nch, k8 = et - sl * nch;
    const bool b_active = sl < nsl;
    const int gc8 = n0 + 8 * k8;                            // global output column of the chunk
    float b8[8], csum[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      b8[k] = (P.mode == 0 && P.bias && b_active && gc8 + k < P.Nout) ? __ldg(P.bias + gc8 + k) : 0.f;
      csum[k] = 0.f;
    }
    int tr = 0;
#define EDG_TRACE() do { if (P.trace && blockIdx.x == 0 && et == 0 && tr < 250) P.trace[tr++] = clock64(); } while (0)
    EDG_TRACE();
    if (pool) for (int i = et; i < kFMaxSent * tabw; i += kEpiThreads) tab[i] = 0u;
    for (int i = et; i < pitch / 4; i += kEpiThreads)             // the zero row: target of the unused neighbour slots
      reinterpret_cast<uint32_t*>(sm + P.off_s + (size_t)P.rows_cap * pitch)[i] = 0u;
    epi_bar(kEpiThreads);
    // patch entries (adjoint): global arg-max row and value per (sentence of the tile, this thread's column)
    float pv[kFMaxSent];
    int pg[kFMaxSent];
    auto load_patch = [&](const int32_t* h) {
      const int s0_ = h[3], ns_ = h[2];
      const int gc = n0 + et;
#pragma unroll
      for (int s = 0; s < kFMaxSent; ++s) {
        pv[s] = 0.f; pg[s] = -1;
        if (et < cw && gc < P.Nout && s < ns_) {
          const int64_t o = (int64_t)(s0_ + s) * P.ldpatch + gc;
          pg[s] = __ldg(P.patch_arg + o);
          pv[s] = __ldg(P.patch_val + o);
        }
      }
    };
    if (patch && t_first < n_tiles) {
      f2_wait(cfull(0), 0);
      load_patch(reinterpret_cast<const int32_t*>(sm + P.off_csr));
    }
    int it = 0;
    for (int t = t_first; t < n_tiles; t += t_step, ++it) {
      const int as = it % kFAccStages;
      const uint32_t aphase = (uint32_t)(it / kFAccStages) & 1u;
      const int cb = it % kFCsrBufs;
      const uint32_t cphase = (uint32_t)(it / kFCsrBufs) & 1u;
      const uint32_t cs_s = base + P.off_csr + cb * kFCsrBytes;
      const uint8_t* cs = sm + P.off_csr + cb * kFCsrBytes;
      const int32_t* hdr = reinterpret_cast<const int32_t*>(cs);
      const uint8_t* sfirst = cs + 16;
      const uint32_t meta_s = cs_s + 32;
      EDG_TRACE();
      f2_wait(cfull(cb), cphase);
      EDG_TRACE();
      const int r0 = hdr[0], n = hdr[1], ns = hdr[2], s0 = hdr[3];
      // ---- patch entries of the tile: thread = column, one entry per sentence (tile-local u8 rows, 0xff = none); the
      // global loads were issued one tile ahead (below), so no DRAM round trip is waited for here
      uint32_t pa_lo = 0xffffffffu, pa_hi = 0xffffffffu;
      if (patch) {
#pragma unroll
        for (int s = 0; s < kFMaxSent; ++s) {
          const int a = pg[s] - r0;
          const uint32_t lr = (pg[s] >= 0 && a >= 0 && a < n) ? (uint32_t)a : 0xffu;
          if (s < 4) pa_lo = (pa_lo & ~(0xffu << (8 * s))) | (lr << (8 * s));
          else pa_hi = (pa_hi & ~(0xffu << (8 * (s - 4)))) | (lr << (8 * (s - 4)));
        }
      }
      f2_wait(tfull(as), aphase);
      EDG_TRACE();
      tc_fence_after();
      const uint32_t tbase = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(as * kFAccStride);
      const int row = q * 32 + lane;
      const bool row_ok = row < n;
      float scale = 1.f;
      if (P.mode == 1 && row_ok) {
        uint32_t my;
        asm volatile("ld.shared.u32 %0, [%1];" : "=r"(my) : "r"(meta_s + 16u * row + 8u));
        scale = lut[my & 0xffu];
      }
      // ---- phase A: accumulator -> (adjoint: x 1/(deg+1)) -> bf16 staging; thread = row, 16-column granules
      if (q * 32 < n && !(P.debug & 2)) {
        const uint32_t srow_addr = s_base + (uint32_t)(row * pitch);
        const int ngran = cw >> 4;
        uint32_t ra[16], rb[16];
        auto stage_out = [&](const uint32_t (&r)[16], int g) {
          if (row_ok) {
            uint32_t w[8];
#pragma unroll
            for (int k = 0; k < 8; ++k) w[k] = pack_bf16x2(__uint_as_float(r[2 * k]) * scale, __uint_as_float(r[2 * k + 1]) * scale);
            st_shared_v4(srow_addr + (uint32_t)(g * 32), w[0], w[1], w[2], w[3]);
            st_shared_v4(srow_addr + (uint32_t)(g * 32 + 16), w[4], w[5], w[6], w[7]);
          }
        };
        int g = part;
        if (g < ngran) tmem_ld_32x32_x16(tbase + g * 16, ra);
        while (g < ngran) {
          tmem_wait_ld();
          const int g1 = g + nparts;
          if (g1 < ngran) tmem_ld_32x32_x16(tbase + g1 * 16, rb);
          stage_out(ra, g);
          g = g1;
          if (g >= ngran) break;
          tmem_wait_ld();
          const int g2 = g + nparts;
          if (g2 < ngran) tmem_ld_32x32_x16(tbase + g2 * 16, ra);
          stage_out(rb, g);
          g = g2;
        }
      }
      tc_fence_before();                                     // accumulator drained: the MMA warp may reuse the stage
      __syncwarp();
      if (lane == 0) mbar_arrive(tempty(as));
      epi_bar(kEpiThreads);
      EDG_TRACE();
      // ---- patch (adjoint): staging[arg][c] += val / (deg_arg + 1); thread = column: distinct addresses
      if (patch) {
        if (et < cw) {
#pragma unroll
          for (int s = 0; s < kFMaxSent; ++s) {
            const uint32_t lr = ((s < 4 ? pa_lo : pa_hi) >> (8 * (s & 3))) & 0xffu;
            if (lr != 0xffu) {
              uint32_t my;
              asm volatile("ld.shared.u32 %0, [%1];" : "=r"(my) : "r"(meta_s + 16u * lr + 8u));
              __nv_bfloat16* dst = reinterpret_cast<__nv_bfloat16*>(sm + P.off_s + (size_t)lr * pitch) + et;
              *dst = __float2bfloat16_rn(__bfloat162float(*dst) + pv[s] * lut[my & 0xffu]);
            }
          }
        }
        epi_bar(kEpiThreads);
        if (t + t_step < n_tiles) {                          // the next tile's entries: in flight during phase B
          const int cbn = (it + 1) % kFCsrBufs;
          f2_wait(cfull(cbn), (uint32_t)((it + 1) / kFCsrBufs) & 1u);
          load_patch(reinterpret_cast<const int32_t*>(sm + P.off_csr + cbn * kFCsrBytes));
        }
      }
      // ---- phase B: y_i = sum of the staged rows of i's neighbours; one 16-byte load per neighbour slot
      if (b_active) {
        const uint32_t aT = s_base + (uint32_t)k8 * 16u;
        const bool col_ok = gc8 + 8 <= (int)P.ldy;
        int cur_s = -1;
        uint32_t vmax[4] = {0u, 0u, 0u, 0u}, varg[4] = {0u, 0u, 0u, 0u};     // packed bf16x2 maxima / u16x2 rows
        auto flush = [&]() {
#pragma unroll
          for (int w = 0; w < 4; ++w) {
            const int cbase = cur_s * tabw + 8 * k8 + 2 * w;
            atomicMax(tab + cbase, pool_key(vmax[w] << 16, 0xffffu - (varg[w] & 0xffffu)));
            atomicMax(tab + cbase + 1, pool_key(vmax[w], 0xffffu - (varg[w] >> 16)));
          }
        };
        // a slice owns a CONTIGUOUS block of rows: it then crosses a sentence boundary (= one flush of eight shared-memory
        // atomics) once or twice per tile instead of once per sentence of the tile
        const int rps = (n + nsl - 1) / nsl;                  // rows per slice
        const int i_beg = sl * rps, i_end = (P.debug & 1) ? 0 : min(n, i_beg + rps);
        __nv_bfloat16* yp = P.y + (int64_t)(r0 + i_beg) * P.ldy + gc8;
        const int64_t ystep = P.ldy;
        uint32_t m0 = 0, m1 = 0, m2 = 0, m3 = 0;
        if (i_beg < n) asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(m0), "=r"(m1), "=r"(m2), "=r"(m3) : "r"(meta_s + 16u * i_beg));
#pragma unroll 1
        for (int i = i_beg; i < i_end; ++i, yp += ystep) {
          const uint32_t nb_lo = m0, nb_hi = m1, info = m2, e_glob = m3;
          const int deg = info & 0xffu, s = (info >> 8) & 0xffu;
          if (i + 1 < i_end)
            asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(m0), "=r"(m1), "=r"(m2), "=r"(m3) : "r"(meta_s + 16u * (i + 1)));
          float inv;
          asm volatile("ld.shared.f32 %0, [%1];" : "=f"(inv) : "r"(lut_s + 4u * deg));
          uint32_t v[4][4];
#pragma unroll
          for (int u = 0; u < 4; ++u) {                      // self + three neighbours (unused slots read the zero row)
            const uint32_t ro = ((nb_lo >> (8 * u)) & 0xffu) * (uint32_t)pitch;
            asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v[u][0]), "=r"(v[u][1]), "=r"(v[u][2]), "=r"(v[u][3]) : "r"(aT + ro));
          }
          float acc[8];
#pragma unroll
          for (int w = 0; w < 4; ++w) {                      // FHADD.BF16: no unpack instructions (edg_common.cuh)
            acc[2 * w] = __uint_as_float(v[0][w] << 16);
            acc[2 * w + 1] = __uint_as_float(v[0][w] & 0xffff0000u);
#pragma unroll
            for (int u = 1; u < 4; ++u) add_bf16x2(v[u][w], acc[2 * w], acc[2 * w + 1]);
          }
          if (deg > 4) {                                     // one row in eight: four more slots
            uint32_t x[4][4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              const uint32_t ro = ((nb_hi >> (8 * u)) & 0xffu) * (uint32_t)pitch;
              asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(x[u][0]), "=r"(x[u][1]), "=r"(x[u][2]), "=r"(x[u][3]) : "r"(aT + ro));
            }
#pragma unroll
            for (int w = 0; w < 4; ++w)
#pragma unroll
              for (int u = 0; u < 4; ++u) add_bf16x2(x[u][w], acc[2 * w], acc[2 * w + 1]);
            if (deg > 8) {                                   // hubs: the rest of the row's entries from the global CSR
              int cnt = 0;
              for (int e = 0; e < deg; ++e) {
                const int j = __ldg(P.col + e_glob + e) - r0;
                if (j == i) continue;
                if (cnt++ < 7) continue;
                uint32_t z[4];
                asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(z[0]), "=r"(z[1]), "=r"(z[2]), "=r"(z[3]) : "r"(aT + (uint32_t)j * (uint32_t)pitch));
#pragma unroll
                for (int w = 0; w < 4; ++w) add_bf16x2(z[w], acc[2 * w], acc[2 * w + 1]);
              }
            }
          }
          if (P.mode == 1) {                                 // column sums of the raw rows: un-scale the self term
            const float wgt = (float)(deg + 1);
#pragma unroll
            for (int w = 0; w < 4; ++w) {
              csum[2 * w] = fmaf(__uint_as_float(v[0][w] << 16), wgt, csum[2 * w]);
              csum[2 * w + 1] = fmaf(__uint_as_float(v[0][w] & 0xffff0000u), wgt, csum[2 * w + 1]);
            }
          } else {
#pragma unroll
            for (int k = 0; k < 8; ++k) acc[k] = fmaf(acc[k], inv, b8[k]);
          }
          uint32_t pw[4];
#pragma unroll
          for (int w = 0; w < 4; ++w) pw[w] = pack_bf16x2(acc[2 * w], acc[2 * w + 1]);
          if (col_ok) *reinterpret_cast<uint4*>(yp) = make_uint4(pw[0], pw[1], pw[2], pw[3]);
          if (pool) {
            // running column maxima on packed bf16 pairs: strict > keeps the FIRST row on ties (torch.max)
            const uint32_t ipk = (uint32_t)i * 0x00010001u;
            if (s != cur_s) {
              if (cur_s >= 0) flush();
              cur_s = s;
#pragma unroll
              for (int w = 0; w < 4; ++w) { vmax[w] = pw[w]; varg[w] = ipk; }
            } else {
#pragma unroll
              for (int w = 0; w < 4; ++w) {
                const __nv_bfloat162 nv = *reinterpret_cast<const __nv_bfloat162*>(&pw[w]);
                const __nv_bfloat162 ov = *reinterpret_cast<const __nv_bfloat162*>(&vmax[w]);
                const uint32_t gt = __hgt2_mask(nv, ov);
                const __nv_bfloat162 mx = __hmax2(ov, nv);
                vmax[w] = *reinterpret_cast<const uint32_t*>(&mx);
                varg[w] = (varg[w] & ~gt) | (ipk & gt);
              }
            }
          }
        }
        if (pool && cur_s >= 0) flush();
      }
      epi_bar(kEpiThreads);
      EDG_TRACE();
      // ---- pool table -> global (and reset): thread = column; the next writers of the table come after another barrier
      if (pool && et < cw) {
        const int gc = n0 + et;
        for (int s = 0; s < ns; ++s) {
          const uint32_t key = tab[s * tabw + et];
          tab[s * tabw + et] = 0u;
          if (gc < P.Nout) {
            const int64_t o = (int64_t)(s0 + s) * P.ldpool + gc;
            const bool any = sfirst[s + 1] > sfirst[s];
            P.hmax[o] = any ? pool_key_value(key) : 0.f;
            P.harg[o] = any ? r0 + (int)(0xffffu - (key & 0xffffu)) : -1;
          }
        }
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(cempty(cb));
    }
    EDG_TRACE();
#undef EDG_TRACE
    // ---- partial column sums of this CTA (adjoint): reduce the row slices through the staging buffer
    if (P.colsum_part) {
      epi_bar(kEpiThreads);
      float* red = reinterpret_cast<float*>(sm + P.off_s);
      if (b_active) {
#pragma unroll
        for (int k = 0; k < 8; ++k) red[sl * cw + 8 * k8 + k] = csum[k];
      }
      epi_bar(kEpiThreads);
      for (int c = et; c < cw; c += kEpiThreads) {
        float a = 0.f;
        for (int s = 0; s < nsl; ++s) a += red[s * cw + c];
        const int gc = n0 + c;
        if (gc < P.Nout) P.colsum_part[(int64_t)t_first * P.Nout + gc] = a;
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// ---------------------------------------------------------------------------------------------
// tile plan: greedy packing of whole sentences into tiles of <= max_rows rows, <= kFMaxSent sentences and
// <= kFMaxNnz CSR entries.  One block; the chain of tile starts is walked by one thread over u8 jump lengths
// in shared memory (~30 cycles per tile).
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024)
tile_plan_kernel(const int32_t* __restrict__ sent_ptr, const int32_t* __restrict__ row_ptr, int B, int max_rows,
                 int32_t* __restrict__ info, int32_t* __restrict__ n_tiles) {
  extern __shared__ uint8_t jump[];                 // [B] sentences in the tile that starts at s
  __shared__ int nt_s;
  for (int s = threadIdx.x; s < B; s += blockDim.x) {
    const int rs = __ldg(sent_ptr + s);
    const int es = __ldg(row_ptr + rs);
    int lo = s + 1, hi = min(B, s + kFMaxSent);      // largest e in [lo, hi] that still fits (e = s + 1 always taken)
    while (lo < hi) {
      const int mid = (lo + hi + 1) >> 1;
      const int rm = __ldg(sent_ptr + mid);
      const bool ok = (rm - rs <= max_rows) && (__ldg(row_ptr + rm) - es <= kFMaxNnz);
      if (ok) lo = mid; else hi = mid - 1;
    }
    jump[s] = (uint8_t)(lo - s);
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    int s = 0, t = 0;
    while (s < B) { info[8 * t] = s; s += jump[s]; ++t; }
    nt_s = t;
    *n_tiles = t;
  }
  __syncthreads();
  const int nt = nt_s;
  for (int t = threadIdx.x; t < nt; t += blockDim.x) {
    const int s0 = info[8 * t];
    const int s1 = s0 + jump[s0];
    const int r0 = __ldg(sent_ptr + s0), r1 = __ldg(sent_ptr + s1);
    info[8 * t + 1] = s1; info[8 * t + 2] = r0; info[8 * t + 3] = r1;
    info[8 * t + 4] = __ldg(row_ptr + r0); info[8 * t + 5] = __ldg(row_ptr + r1);
    info[8 * t + 6] = 0; info[8 * t + 7] = 0;
  }
}

// out[c] (+)= sum_g part[g][c]: block = 32 columns x 8 partial slices (warp w sums g = w, w + 8, ...), combined through
// shared memory in warp order -- a fixed summation order (deterministic), ~G/8 dependent-free loads per thread
__global__ void __launch_bounds__(256)
colsum_part_reduce_kernel(const float* __restrict__ part, int G, int C, float* __restrict__ out, int accumulate) {
  __shared__ float red[8][32];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int c = blockIdx.x * 32 + lane;
  float a = 0.f;
  if (c < C)
    for (int g = w; g < G; g += 8) a += part[(int64_t)g * C + c];
  red[w][lane] = a;
  __syncthreads();
  if (w == 0 && c < C) {
    float t = red[0][lane];
#pragma unroll
    for (int k = 1; k < 8; ++k) t += red[k][lane];
    out[c] = accumulate ? out[c] + t : t;
  }
}

// Backward of the gated max-pool views of layer 1 and the diversity term (bert_amir5.py:627-638) from the column
// maxima the fused layer kernel returns: pooled_v = g_v * hmax (the views share their arg-max row for positive gates),
// d xy / d pooled_v = g_xy / B * sum_{v' != v} pooled_v'.  Writes what the arg-max rows of d h_1 receive (patch_val,
// consumed by edg_gcn_layer mode 1) and the gates' share d g_v = d pooled_v * hmax.
__global__ void __launch_bounds__(256)
views_bwd_hmax_kernel(const float* __restrict__ hmax, const float* __restrict__ gates, const float* __restrict__ g_xy,
                      int V, int B, int D, float* __restrict__ patch_val, int64_t ldp, float* __restrict__ dgates, int acc_view) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;      // B * D < 2^31 (checked by the caller)
  const int BD = B * D;
  if (i >= BD) return;
  const int b = i / D, d = i - b * D;
  const float gxy = g_xy ? (__ldg(g_xy) / (float)B) : 0.f;
  const float hm = hmax[i];
  float gsum = 0.f;
  for (int v = 0; v < V; ++v) gsum += gates[v * BD + i];
  float pval = 0.f;
  for (int v = 0; v < V; ++v) {
    const float g = gates[v * BD + i];
    const float dp = gxy * (gsum - g) * hm;               // d xy / d pooled_v
    pval = fmaf(dp, g, pval);
    const float dg = dp * hm;
    dgates[v * BD + i] = (v == acc_view) ? dgates[v * BD + i] + dg : dg;
  }
  patch_val[(int64_t)b * ldp + d] = pval;
}

struct FusedPlan { int npass, stages, rows_cap, pitch, bn0, bn1, n_split, epi_warps; size_t smem;
                   uint32_t off_a, off_s, off_tab, off_csr, off_scr, off_lut, off_bar; bool ok; };

static int fused_env(const char* name, int dflt) {
  const char* e = getenv(name);
  return e ? atoi(e) : dflt;
}

// Shared-memory plan: stationary weight slice | K-block ring | bf16 staging tile (+ zero row) | pool table | CSR buffers.
static FusedPlan plan_fused(int K, int Nout) {
  FusedPlan p;
  memset(&p, 0, sizeof(p));
  p.ok = false;
  if (K <= 0 || Nout <= 0 || K > 64 * 5 || Nout > 2 * kFAccStride) return p;
  const int num_kb = (K + 63) / 64;
  const int n16 = (Nout + 15) / 16 * 16;
  if (n16 <= kFAccStride) { p.n_split = 1; p.bn0 = n16; p.bn1 = 0; }
  else { p.n_split = 2; p.bn0 = ((n16 / 2 + 15) / 16) * 16; p.bn1 = n16 - p.bn0; }
  p.npass = 1;
  p.epi_warps = fused_env("EDG_FUSED_EPI_WARPS", 8);
  if (p.epi_warps != 8 && p.epi_warps != 12) p.epi_warps = 8;
  const int cw = p.bn0 / p.npass;
  p.pitch = cw * 2 + 16;                               // bf16 staging; an odd number of 16-byte chunks per row
  const size_t budget = 227 * 1024 - 1024;            // 1 KB for the 1024-byte alignment of the dynamic base
  const size_t w_bytes = (size_t)num_kb * p.bn0 * 128;
  const size_t tab = (size_t)kFMaxSent * cw * 4;
  const size_t min_stage = (size_t)kFMaxEpiWarps * 32 * 8 * 4;        // the column-sum scratch reuses the staging tile
  const size_t fixed = w_bytes + tab + (size_t)kFCsrBufs * kFCsrBytes + 2 * kFScratch + kFLut * 4 + 512 + (size_t)p.pitch;   // + the zero row
  // rows: as many as fit next to >= 3 ring stages, at most 128
  int rows = kFRows;
  int want = fused_env("EDG_FUSED_ROWS", 0);
  if (want >= 32 && want <= kFRows) rows = want;
  while (rows >= 32 && fixed + (size_t)rows * p.pitch + 3 * 16384 > budget) rows -= 2;
  size_t stage_bytes = (size_t)(rows + 1) * p.pitch;
  if (stage_bytes < min_stage) stage_bytes = min_stage;
  if (rows < 32) return p;
  p.rows_cap = rows;
  int stages = (int)((budget - (fixed - p.pitch) - stage_bytes) / 16384);
  if (stages > kFMaxStages) stages = kFMaxStages;
  int ws = fused_env("EDG_FUSED_STAGES", 0);
  if (ws >= 2 && ws < stages) stages = ws;
  p.stages = stages;
  uint32_t off = (uint32_t)w_bytes;                   // W at 0 (1024-aligned blocks: bn * 128 with bn % 16 == 0 -> % 2048)
  off = (off + 1023u) & ~1023u;
  p.off_a = off; off += (uint32_t)stages * 16384u;
  p.off_s = off; off += (uint32_t)stage_bytes;
  off = (off + 15u) & ~15u;
  p.off_tab = off; off += (uint32_t)tab;
  p.off_csr = off; off += kFCsrBufs * kFCsrBytes;
  p.off_scr = off; off += 2 * kFScratch;
  p.off_lut = off; off += kFLut * 4;
  off = (off + 7u) & ~7u;
  p.off_bar = off; off += 512;
  p.smem = (size_t)off + 1024;
  p.ok = p.smem <= 227 * 1024;
  return p;
}

}  // namespace edg

using namespace edg;

/* see include/edgcn.h */
extern "C" int edg_fused_tile_rows(int32_t K, int32_t Nout) {
  const FusedPlan p = plan_fused(K, Nout);
  return p.ok ? p.rows_cap : 0;
}

extern "C" int edg_views_bwd_hmax(const float* hmax, const float* gates, const float* g_xy, int32_t V, int32_t B, int32_t D,
                                  float* patch_val, int64_t ldp, float* dgates, int acc_view, edg_stream stream) {
  if (V <= 0 || B < 0 || D <= 0 || ldp < D) return EDG_ERR_ARG;
  if (B == 0) return EDG_OK;
  if (!hmax || !gates || !patch_val || !dgates) return EDG_ERR_ARG;
  if ((int64_t)B * D * V >= (int64_t)1 << 31) return EDG_ERR_UNSUPPORTED;
  const int64_t total = (int64_t)B * D;
  views_bwd_hmax_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(hmax, gates, g_xy, V, B, D, patch_val, ldp,
                                                                                         dgates, acc_view);
  return check_launch();
}

extern "C" int edg_tile_plan(const int32_t* sent_ptr, const int32_t* row_ptr, int32_t B, int32_t max_rows,
                             int32_t* tile_info, int32_t* n_tiles, edg_stream stream) {
  if (B < 0 || max_rows < 1 || max_rows > kFRows) return EDG_ERR_ARG;
  if (!sent_ptr || !row_ptr || !tile_info || !n_tiles) return EDG_ERR_ARG;
  if (B > 200 * 1024) return EDG_ERR_UNSUPPORTED;
  const size_t smem = (size_t)(B > 0 ? B : 1);
  if (int rc_ = ensure_dyn_smem((const void*)tile_plan_kernel, smem)) return rc_;
  tile_plan_kernel<<<1, 1024, smem, (cudaStream_t)stream>>>(sent_ptr, row_ptr, B, max_rows, tile_info, n_tiles);
  return check_launch();
}

extern "C" int edg_gcn_layer(const void* x, int64_t ldx, int32_t N, int32_t K, const void* w, int64_t ldw, int32_t Nout,
                             const float* bias, int mode, const int32_t* row_ptr, const int32_t* col,
                             const int32_t* sent_ptr, const int32_t* tile_info, const int32_t* n_tiles, int32_t tile_rows,
                             void* y, int64_t ldy, float* hmax, int32_t* harg, int64_t ldpool, const float* patch_val,
                             const int32_t* patch_arg, int64_t ldpatch, float* colsum, int colsum_accumulate, void* ws,
                             size_t ws_bytes, edg_stream stream) {
  if (N < 0 || K <= 0 || Nout <= 0 || (mode != 0 && mode != 1)) return EDG_ERR_ARG;
  if (N == 0) return EDG_OK;
  if (!x || !w || !y || !row_ptr || !col || !sent_ptr || !tile_info || !n_tiles) return EDG_ERR_ARG;
  if ((hmax != nullptr) != (harg != nullptr) || (patch_val != nullptr) != (patch_arg != nullptr)) return EDG_ERR_ARG;
  if (mode == 0 && (patch_val || colsum)) return EDG_ERR_ARG;
  if (mode == 1 && (hmax || bias)) return EDG_ERR_ARG;
  if (ldx < K || ldw < K || ldy < Nout) return EDG_ERR_ARG;
  if (!aligned16(x) || !aligned16(w) || !aligned16(y) || (ldx & 7) || (ldw & 7) || (ldy & 7)) return EDG_ERR_ALIGN;
  cudaStream_t s = (cudaStream_t)stream;
  const FusedPlan p = plan_fused(K, Nout);
  if (!p.ok || tile_rows > p.rows_cap) return EDG_ERR_UNSUPPORTED;
  const int groups = kNumSMs / p.n_split;
  if (colsum && ws_bytes < (size_t)groups * Nout * sizeof(float)) return EDG_ERR_WORKSPACE;
  GcnLayerParams P;
  memset(&P, 0, sizeof(P));
  int box_rows = fused_env("EDG_FUSED_BOXROWS", 32);
  if (box_rows != 32 && box_rows != 64 && box_rows != 128) box_rows = 32;
  P.box_rows = box_rows;
  int rc = make_map_bf16(&P.map_a, x, N, K, ldx, 64, box_rows);
  if (rc) return rc;
  rc = make_map_bf16(&P.map_w, w, Nout, K, ldw, 64, 16);
  if (rc) return rc;
  P.tile_info = tile_info; P.n_tiles = n_tiles; P.row_ptr = row_ptr; P.col = col; P.sent_ptr = sent_ptr;
  P.bias = bias; P.y = (__nv_bfloat16*)y; P.ldy = ldy; P.hmax = hmax; P.harg = harg; P.ldpool = ldpool;
  P.patch_val = patch_val; P.patch_arg = patch_arg; P.ldpatch = ldpatch;
  P.colsum_part = colsum ? (float*)ws : nullptr;
  P.trace = (!colsum && ws && ws_bytes >= 2048 && (fused_env("EDG_FUSED_DEBUG", 0) & 32)) ? (long long*)ws : nullptr;
  P.K = K; P.Nout = Nout; P.num_kb = (K + 63) / 64; P.mode = mode; P.n_split = p.n_split; P.npass = p.npass;
  P.stages = p.stages; P.rows_cap = p.rows_cap; P.debug = fused_env("EDG_FUSED_DEBUG", 0);
  P.bn[0] = p.bn0; P.bn[1] = p.bn1;
  P.idesc[0] = make_idesc_bf16(kFRows, p.bn0, 0, 0);
  P.idesc[1] = make_idesc_bf16(kFRows, p.bn1 > 0 ? p.bn1 : 16, 0, 0);
  P.pitch = p.pitch;
  P.sleep_ns = fused_env("EDG_FUSED_SLEEP", 64);
  P.prefetch = fused_env("EDG_FUSED_PF", 0);       // L2 prefetch of the tiles ahead: measured slower (71 vs 66 us), off
  if (P.prefetch < 0 || P.prefetch > 3) P.prefetch = 0;
  P.off_a = p.off_a; P.off_s = p.off_s; P.off_tab = p.off_tab; P.off_csr = p.off_csr; P.off_scr = p.off_scr; P.off_lut = p.off_lut; P.off_bar = p.off_bar;
  const int grid = groups * p.n_split;
  if (p.epi_warps == 12) {
    if (int rc_ = ensure_dyn_smem((const void*)gcn_layer_kernel<12>, p.smem)) return rc_;
    gcn_layer_kernel<12><<<grid, (4 + 12) * 32, p.smem, s>>>(P);
  } else {
    if (int rc_ = ensure_dyn_smem((const void*)gcn_layer_kernel<8>, p.smem)) return rc_;
    gcn_layer_kernel<8><<<grid, (4 + 8) * 32, p.smem, s>>>(P);
  }
  rc = check_launch();
  if (rc) return rc;
  if (colsum) {
    colsum_part_reduce_kernel<<<(Nout + 31) / 32, 256, 0, s>>>((const float*)ws, groups, Nout, colsum, colsum_accumulate);
    rc = check_launch();
  }
  return rc;
}
