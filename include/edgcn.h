/*
 * edgcn.h -- C ABI of the B200-native gated-GCN hot path (libedgcn.so).
 *
 * This is the drop-in boundary for ONE path of laiviet/ed-gated-gcn: the
 * trigger-conditioned gated graph convolution (SURVEY.md section 8).  The reference
 * is pure Python/PyTorch and has no FFI of its own; each entry point below names
 * the reference lines whose work it replaces (paths relative to the reference
 * repository root).  INTEGRATION.md shows the ctypes binding and the one-line
 * change to models/gcn.py that a reference maintainer would make.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer owned by the caller (torch); the library
 *     allocates nothing and keeps no global state;
 *   - sizes and leading dimensions (ld*) are in ELEMENTS, not bytes;
 *   - `stream` is the cudaStream_t to enqueue on (torch.cuda.current_stream());
 *     calls only enqueue work, they never synchronise;
 *   - return value: EDG_OK (0) or a negative edg_status; nothing throws or
 *     exits across the ABI; asynchronous CUDA faults surface at the caller's
 *     next synchronisation as usual;
 *   - re-entrant and thread-safe (autograd calls backward from another host thread);
 *   - sm_100a only: there is no CPU path and no other-arch path.
 *
 * Layout vocabulary
 *   sentence b owns the packed token rows [sent_ptr[b], sent_ptr[b+1]);
 *   N = total rows, B = sentences (= graphs = (sentence, trigger) pairs);
 *   CSR (row_ptr[N+1], col[nnz]) holds, for row i, the GLOBAL row ids of
 *   self + parent + children in ascending order (the non-zeros of graph.py:66-75);
 *   activations are row-major [N, ld] in fp32 or bf16, rows 16-byte aligned.
 */
#ifndef EDGCN_H_
#define EDGCN_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define EDG_ABI_VERSION 5

typedef enum {
  EDG_OK = 0,
  EDG_ERR_ARG = -1,         /* null pointer, negative size, bad enum            */
  EDG_ERR_ALIGN = -2,       /* pointer or leading dimension not 16-byte aligned */
  EDG_ERR_DTYPE = -3,       /* dtype combination not implemented                */
  EDG_ERR_ARCH = -4,        /* device is not sm_100                             */
  EDG_ERR_WORKSPACE = -5,   /* workspace too small (see the *_workspace query)  */
  EDG_ERR_CUDA = -6,        /* a CUDA runtime/driver call failed at enqueue     */
  EDG_ERR_UNSUPPORTED = -7  /* shape outside what the kernels implement         */
} edg_status;

typedef enum { EDG_F32 = 0, EDG_BF16 = 1 } edg_dtype;
typedef enum { EDG_ACT_NONE = 0, EDG_ACT_SIGMOID = 1, EDG_ACT_RELU = 2 } edg_act;
typedef enum { EDG_PAD_MAX_PLUS_1 = 0, EDG_PAD_ZERO = 1 } edg_pad;
typedef void* edg_stream;   /* cudaStream_t */

int edg_version(void);
const char* edg_strerror(int status);
/* Last CUDA error string recorded by this thread's most recent failing call. */
const char* edg_last_cuda_error(void);

/* ------------------------------------------------------------------------- */
/* Integer kernels (bit-exact against the reference)                          */
/* ------------------------------------------------------------------------- */

/* graph.py:66-75 (gen_graph, matrix part) in packed form.  heads[N] holds the
 * sentence-local head index of every token (-1 = root; out-of-range or self
 * heads are treated as root).  Writes row_ptr[N+1], col (capacity >= 3N),
 * row_sent[N] (sentence id of each row).  ws: B+1 int32 of scratch.
 * max_len = longest sentence (<= 4096). */
int edg_csr_from_heads(const int32_t* heads, const int32_t* sent_ptr, int32_t B, int32_t N,
                       int32_t max_len, int32_t* row_ptr, int32_t* col, int32_t* row_sent,
                       int32_t* ws, edg_stream stream);

/* graph.py:66-75 for graphs that are not forests (CoreNLP enhanced dependencies,
 * graph.py:63-64): the forest of heads[] (as in edg_csr_from_heads) plus E extra
 * undirected edges.  edges[E][2] holds sentence-local (i, j) pairs; sentence b owns
 * pairs edge_ptr[b] .. edge_ptr[b+1]-1 (edge_ptr[B+1], edge_ptr[0] = 0, edge_ptr[B] = E).
 * Set semantics: duplicate pairs, both orientations of one pair, pairs that repeat a
 * forest edge and i == j change nothing; a pair with an endpoint outside [0, n_b) is
 * dropped.  Each row lists self, parent, children and extra neighbours once, as
 * global ids in ascending order, so the output does not depend on the order of the
 * pairs.  Writes row_ptr[N+1], col (capacity >= 3N + 2E), row_sent[N] and
 * sent_max_nnz[0] = the largest CSR entry count of one sentence.  On entry,
 * sent_max_nnz[0] > 0 is an upper bound the caller guarantees for that count (a
 * sentence above it traps, as one longer than max_len does); 0 = no bound.
 * ws: edg_csr_from_heads_edges_workspace(B, N, E) bytes.  max_len <= 4096; any
 * number of pairs per sentence.  Enqueues 3 kernels when E = 0 or N = 0, 7 otherwise. */
size_t edg_csr_from_heads_edges_workspace(int32_t B, int32_t N, int32_t E);
int edg_csr_from_heads_edges(const int32_t* heads, const int32_t* sent_ptr, const int32_t* edges,
                             const int32_t* edge_ptr, int32_t B, int32_t N, int32_t E, int32_t max_len,
                             int32_t* row_ptr, int32_t* col, int32_t* row_sent, int32_t* sent_max_nnz,
                             void* ws, size_t ws_bytes, edg_stream stream);

/* Compat path for the unchanged forward(text, adj) signature (models/gcn.py:30):
 * dense [B,T,T] adjacency (fp32 or int64, any strides) -> packed CSR over B*T rows
 * (padding rows are self-loop singletons, graph.py:66).  Two calls because the
 * caller must size `col`: _count fills row_ptr[B*T+1] (nnz = row_ptr[B*T]) and
 * flags[0] = entries that are neither 0 nor 1, flags[1] = asymmetric entries;
 * _fill writes col. */
int edg_csr_from_dense_count(const void* adj, int adj_is_i64, int32_t B, int32_t T,
                             int64_t stride_b, int64_t stride_r, int64_t stride_c,
                             int32_t* row_ptr, int32_t* flags, edg_stream stream);
int edg_csr_from_dense_fill(const void* adj, int adj_is_i64, int32_t B, int32_t T,
                            int64_t stride_b, int64_t stride_r, int64_t stride_c,
                            const int32_t* row_ptr, int32_t* col, edg_stream stream);

/* data_utils.py:302-323 (get_dist / get_dist_to_target): hop count from every
 * token to the trigger + 1 (trigger -> 1); a token that cannot reach the trigger
 * gets 100001.  anchor[B] is sentence-local.  dist[N] is packed. */
int edg_tree_dist(const int32_t* row_ptr, const int32_t* col, const int32_t* sent_ptr,
                  const int32_t* anchor, int32_t B, int32_t max_len, int32_t* dist,
                  edg_stream stream);

/* data_utils.py:486-488 (pad with max+1) / :593-594 (pad with 0): packed
 * distances -> int64 [B,T] as collate_fn lays them out (data_utils.py:378). */
int edg_dist_pad(const int32_t* dist, const int32_t* sent_ptr, int32_t B, int32_t T,
                 int pad_mode, int64_t* out, edg_stream stream);

/* ------------------------------------------------------------------------- */
/* Graph convolution (models/gcn.py:30-45)                                    */
/* ------------------------------------------------------------------------- */

/* Degree-normalised neighbour aggregation, the `adj @ . / (rowsum + 1)` half of
 * gcn.py:35,41 on the packed CSR.
 *   mode 0 (forward):  y[i] = 1/(deg_i+1) * sum_{j in row i} x[j]
 *   mode 1 (backward): y[j] = sum_{i in row j} x[i] / (deg_i+1)   (A symmetric)
 * x and y may differ in dtype; accumulation is fp32.
 * sent_ptr[B+1], row_sent[N] and max_len (longest sentence) enable the shared-memory staged
 * kernel (rows of whole sentences are bulk-copied into shared memory once and gathered from
 * there); pass NULL/0 to gather straight from global memory. */
int edg_aggregate(const void* x, int x_dtype, int64_t ldx, void* y, int y_dtype, int64_t ldy,
                  int32_t N, int32_t D, const int32_t* row_ptr, const int32_t* col, int mode,
                  const int32_t* sent_ptr, const int32_t* row_sent, int32_t B, int32_t max_len,
                  edg_stream stream);

/* One graph-convolution layer as ONE kernel (projection on tcgen05, the degree-normalised aggregation of the
 * sentence tree and the gated max-pool in its epilogue), replacing the matmul + bmm + divide + bias of
 * models/gcn.py:33-45 and the torch.max pools of bert_amir5.py:627-640 without materialising `adj @ hidden`:
 *   mode 0 (forward):  y = A^ (x W^T) + bias,        A^ = D^-1 A   (the reference's own association, gcn.py:34-41)
 *                      hmax[b,d] = max_t y[t,d] over the sentence's rows (of the bf16-rounded y), harg = the GLOBAL row
 *                      of that maximum, first row on ties (torch.max), -1 for an empty sentence       (both optional)
 *   mode 1 (adjoint):  y = A^T (x W^T + patch),      patch[patch_arg[b,d], d] = patch_val[b,d]  (optional: the
 *                      gradient the pooled views of bert_amir5.py:627-638 route to their arg-max rows; patch_arg < 0 =
 *                      none); colsum[d] (+)= column sums of (x W^T + patch)  (optional: the bias gradient of the layer
 *                      below).  With u_l = h_{l-1} W_l the backward pass of layer l is du_l = A^T dh_l,
 *                      dW_l = h_{l-1}^T du_l, dh_{l-1} = du_l W_l^T, so x = du_l, w = W_l gives y = du_{l-1}.
 * x bf16 [N, ldx], w bf16 [Nout, ldw] (row n = the weights producing output column n, K contiguous), y bf16
 * [N, ldy], bias fp32.  K, Nout <= 320.  Rows are processed in tiles of whole sentences (edg_tile_plan with
 * max_rows <= edg_fused_tile_rows(K, Nout)); every sentence must fit a tile and hold <= 512 CSR entries
 * (a tree of n tokens has 3n - 2).  ws: 148 * Nout floats when colsum is given.  bf16 only (EDG_ERR_UNSUPPORTED
 * outside these limits: callers then run edg_aggregate + edg_linear). */
int edg_fused_tile_rows(int32_t K, int32_t Nout);
/* Backward of the gated max-pool views of layer 1 + the diversity term (bert_amir5.py:627-638) from the column maxima
 * hmax [B,D] that edg_gcn_layer returns (pooled_v = gates[v] * hmax; the views share their arg-max row):
 *   patch_val[b,d] = sum_v gates[v,b,d] * dP_v,   dgates[v,b,d] (+)= dP_v * hmax[b,d]   (+= for v == acc_view, else =)
 * with dP_v = g_xy / B * sum_{v' != v} pooled_v'.  patch_val (pitch ldp) + the harg of edg_gcn_layer are the patch
 * arguments of the mode-1 call that produces d h_1.  g_xy: device scalar (NULL = 0). */
int edg_views_bwd_hmax(const float* hmax, const float* gates, const float* g_xy, int32_t V, int32_t B, int32_t D,
                       float* patch_val, int64_t ldp, float* dgates, int acc_view, edg_stream stream);
/* Greedy packing of whole sentences into tiles of <= max_rows rows (<= 6 sentences, <= 512 CSR entries):
 * tile_info int32 [B+1][8] = {s0, s1, r0, r1, e0, e1, 0, 0} (sentence, row and CSR-entry ranges), n_tiles = device
 * scalar.  One small kernel, no host synchronisation. */
int edg_tile_plan(const int32_t* sent_ptr, const int32_t* row_ptr, int32_t B, int32_t max_rows,
                  int32_t* tile_info, int32_t* n_tiles, edg_stream stream);
int edg_gcn_layer(const void* x, int64_t ldx, int32_t N, int32_t K, const void* w, int64_t ldw, int32_t Nout,
                  const float* bias, int mode, const int32_t* row_ptr, const int32_t* col,
                  const int32_t* sent_ptr, const int32_t* tile_info, const int32_t* n_tiles, int32_t tile_rows,
                  void* y, int64_t ldy, float* hmax, int32_t* harg, int64_t ldpool, const float* patch_val,
                  const int32_t* patch_arg, int64_t ldpatch, float* colsum, int colsum_accumulate, void* ws,
                  size_t ws_bytes, edg_stream stream);

/* C[M,Nout] = act(A[M,K] * W^T + bias), W given as [Nout,K] with K contiguous
 * (nn.Linear layout).  Replaces torch.matmul(text, weight) of gcn.py:34 (with a
 * transposed weight copy) and the nn.Linear calls of the gate MLPs
 * (bert_amir5.py:562-571).  bf16 inputs run on tcgen05 tensor cores fed by TMA;
 * fp32 inputs run an FFMA kernel (fp32-parity mode).  bias is fp32 or NULL. */
int edg_linear(const void* A, int ab_dtype, int64_t lda, int32_t M, int32_t K,
               const void* W, int64_t ldw, int32_t Nout, const float* bias, int act,
               void* C, int c_dtype, int64_t ldc, edg_stream stream);

/* dW[K1,K2] (+)= A[R,K1]^T * B[R,K2]  (fp32 result).  Replaces autograd's weight
 * gradients of gcn.py:34 and of the gate Linears.  bias_of: 0 none, 1 column
 * sums of A, 2 column sums of B -> dbias.  ws: edg_wgrad_workspace() bytes.
 * accumulate != 0 adds into dW/dbias instead of overwriting. */
size_t edg_wgrad_workspace(int32_t R, int32_t K1, int32_t K2, int dtype);
int edg_wgrad(const void* A, int64_t lda, int32_t K1, const void* B, int64_t ldb, int32_t K2,
              int dtype, int32_t R, float* dW, int64_t lddw, float* dbias, int bias_of,
              int accumulate, void* ws, size_t ws_bytes, edg_stream stream);

/* n (<= 8) same-shaped weight gradients dW[i][K1,K2] = A[i][R,K1]^T * B[i][R,K2] (+ dbias[i], bias_of as in
 * edg_wgrad) in ONE launch + one reduction: the Linears of the gate MLPs.  bf16 operands only (EDG_ERR_DTYPE
 * otherwise: use edg_wgrad per problem).  A, B, dW, dbias are HOST arrays of device pointers; all problems
 * share lda / ldb / lddw.  Results are overwritten.  ws: edg_wgrad_batch_workspace() bytes. */
size_t edg_wgrad_batch_workspace(int32_t n, int32_t R, int32_t K1, int32_t K2);
int edg_wgrad_batch(int32_t n, const void* const* A, int64_t lda, int32_t K1, const void* const* B, int64_t ldb,
                    int32_t K2, int dtype, int32_t R, float* const* dW, int64_t lddw, float* const* dbias,
                    int bias_of, void* ws, size_t ws_bytes, edg_stream stream);

/* The gate MLPs (bert_amir5.py:562-571, :621-622) as one launch per direction: n_groups (<= 4) independent
 * chains (one per gate) of n_stages (<= 3) Linear(D,D) layers over the same M rows, D <= 320, bf16 tensor
 * cores with fp32 accumulation; the activation tile never leaves shared memory between the Linears.
 *   mode 0 (forward):  A_{s+1} = sigmoid(A_s W_s^T + bias_s)
 *   mode 1 (backward): A_{s+1} = (A_s W_s^T) * y_s (1 - y_s)     (y_s = NULL: no factor)
 * a0[g]: bf16 [M, lda] input of chain g.  stages: HOST array [n_groups * n_stages] (group-major):
 *   w    bf16 [D, ldw], row n = the weights producing output column n, K contiguous (forward: nn.Linear
 *        weight [out,in]; backward: its transpose [in,out]);
 *   bias fp32 [D] or NULL (forward);  y bf16 [M, ldy] or NULL (backward);
 *   out  global copy of the stage output, bf16 or fp32 [M, ldo], or NULL; bf16 copies get zero padding columns.
 * Returns EDG_ERR_UNSUPPORTED for shapes outside these limits (callers then run edg_linear per layer). */
typedef struct {
  const void* w;
  int64_t ldw;
  const float* bias;
  const void* y;
  int64_t ldy;
  void* out;
  int64_t ldo;
  int out_dtype;
} edg_chain_stage;
int edg_mlp_chain(int mode, int32_t n_groups, int32_t n_stages, const void* const* a0, int64_t lda,
                  const edg_chain_stage* stages, int32_t M, int32_t D, edg_stream stream);

/* fp32 [R,C] master weight -> compute-dtype copy, optionally transposed, padding
 * columns up to ldd zero-filled. */
int edg_cast_2d(const float* src, int64_t lds, int32_t R, int32_t C, void* dst, int dst_dtype,
                int64_t ldd, int transpose, edg_stream stream);

/* The same for up to 32 weights in ONE launch (all compute-dtype copies a training step needs).
 * The arrays are HOST arrays of length n (device pointers inside src/dst). */
int edg_cast_batch(int32_t n, const void* const* src, void* const* dst, const int32_t* R, const int32_t* C,
                   const int64_t* lds, const int64_t* ldd, const int32_t* transpose, int dst_dtype,
                   edg_stream stream);

/* ------------------------------------------------------------------------- */
/* Gated block (models/bert_amir5.py:615-648)                                 */
/* ------------------------------------------------------------------------- */

/* bert_amir5.py:604-605,615-618: the trigger row of every sentence.
 * raw[B,D] fp32 = x[sent_ptr[b]+anchor[b]]; act (compute dtype, ld = ldact) =
 * sigmoid(raw) when lead_sigmoid else raw (first op of the gate MLP, :562). */
int edg_trigger_gather(const void* x, int dtype, int64_t ldx, const int32_t* sent_ptr,
                       const int32_t* anchor, int32_t B, int32_t D, float* raw, void* act,
                       int64_t ldact, int lead_sigmoid, edg_stream stream);
/* backward of the gather: dx[sent_ptr[b]+anchor[b]] += da[b] + sum_k extra[k][b]  (rows are distinct).  da fp32 [B,D] or
 * NULL; extra = n_extra further fp32 [B,D] terms stored one after the other (the gate MLPs' input gradients), or NULL. */
int edg_trigger_scatter_add(const float* da, const float* extra, int32_t n_extra, int32_t B, int32_t D,
                            const int32_t* sent_ptr, const int32_t* anchor, void* dx, int dtype, int64_t lddx,
                            edg_stream stream);

/* bert_amir5.py:627-636,640: pooled[v,b,:] = max_t h[t,:]*gates[v,b,:] over the
 * sentence's rows, arg = global row of the maximum (first row wins ties).
 * An empty sentence (0 rows) gets pooled 0, arg -1 and hmax 0.
 * row_sent[N] + max_len (may be NULL/0) enable the shared-memory staged kernel: the rows of the sentences
 * starting in a window are brought in by one bulk async copy instead of one dependent load per row;
 * the same holds for edg_scores_kl_fwd and edg_head_bwd.
 * hmax (optional, fp32 [B,D]): the plain column maximum max_t h[t,:] of every sentence -- h at the arg-max row,
 * from which the views' forward and backward follow for positive gates (edg_views_bwd_hmax, edg_views_bwd_hmax_pairs). */
int edg_pool_fwd(const void* h, int dtype, int64_t ldh, const int32_t* sent_ptr, int32_t B,
                 int32_t D, const float* gates, int32_t V, float* pooled, int32_t* arg,
                 const int32_t* row_sent, int32_t N, int32_t max_len, float* hmax, edg_stream stream);

/* bert_amir5.py:638: xy = sum_{v<v'} mean_b sum_d pooled[v]*pooled[v'].
 * ws: 1024 floats. */
int edg_diversity_fwd(const float* pooled, int32_t V, int32_t B, int32_t D, float* xy, float* ws,
                      edg_stream stream);

/* backward of the pooled views and the diversity term: with
 * dp[v] = g_xy/B * sum_{v'!=v} pooled[v'] (+ g_pooled[v] when given),
 *   dh[arg[v,b,d], d] += dp[v,b,d]*gates[v,b,d]   (added into dh)
 *   dgates[v,b,d]      = dp[v,b,d]*h[arg[v,b,d], d]   (added to the existing value for v == acc_view,
 *                        which already holds d gate_L from edg_head_bwd; -1 = overwrite everywhere)
 * g_xy is a device scalar (NULL = 0). */
int edg_views_bwd(const float* pooled, const int32_t* arg, const float* gates, const void* h,
                  int dtype, int64_t ldh, int32_t V, int32_t B, int32_t D, const float* g_xy,
                  const float* g_pooled, void* dh, int64_t lddh, float* dgates, int acc_view,
                  edg_stream stream);

/* bert_amir5.py:645-648 in collapsed form (SURVEY A9):
 *   scores[i] = sum_d h[i,d]*gate[b,d]*v[b,d] + c[b]
 *   kl_b[b]   = sum_t softmax_t(scores)*softmax_t(float(dist))
 * dist is packed int32 (dist_i64 = 0) or int64.
 * Optional (NULL to skip): dv_unit[B,D], dc_unit[B] = d kl / d v, d kl / d c per unit upstream
 * gradient, so that the backward pass needs no extra sweep over h when only kl carries gradient; with them (optional)
 * u_unit[N] = d kl / d scores[i] = P_i (Q_i - kl_b) / B and sf_unit[B,D] = sum_t u_t h[t,:] (dv_unit without the gate),
 * the per-row scalars and per-sentence vectors edg_head_du builds the top layer's gradient from.
 * An empty sentence (0 rows) gets kl_b 0, and dv_unit, dc_unit, sf_unit 0. */
int edg_scores_kl_fwd(const void* h, int dtype, int64_t ldh, const int32_t* sent_ptr, int32_t B,
                      int32_t D, const float* gate, const float* v, const float* c,
                      const void* dist, int dist_i64, float* scores, float* kl_b,
                      float* dv_unit, float* dc_unit, float* u_unit, float* sf_unit,
                      const int32_t* row_sent, int32_t N, int32_t max_len, edg_stream stream);

/* edg_views_bwd in halves: parts & 1 = the additions into dh only (h, dgates may be NULL), parts & 2 = dgates only
 * (dh may be NULL).  The halves have different consumers (layer 1's backward / the gate MLPs' backward): two launches
 * on two streams take the dgates half off the critical path. */
int edg_views_bwd_parts(const float* pooled, const int32_t* arg, const float* gates, const void* h,
                        int dtype, int64_t ldh, int32_t V, int32_t B, int32_t D, const float* g_xy,
                        const float* g_pooled, void* dh, int64_t lddh, float* dgates, int acc_view, int parts,
                        edg_stream stream);

/* backward of x_out = gate*h_L through scores/kl, the final max-pool and an
 * optional direct gradient on x_out:
 *   ds[i]   = g_kl/B * P_i*(Q_i - kl_b) + g_scores[i]
 *   dh[i,d] = gate*( ds[i]*v + [i==arg[b,d]]*g_pooled[b,d] + g_xout[i,d] )
 *   dgate[b,d] = sum_t h*( ds*v + [..]*g_pooled + g_xout ),  dv[b,d] = sum_t ds*h*gate,
 *   dc[b] = sum_t ds.
 * g_kl: device scalar or NULL; g_scores, g_pooled, g_xout may be NULL.
 * dh/dgate may be NULL (first pass: only dv/dc, which the host needs before it can
 * back-propagate through the classifier head to obtain g_pooled).
 * max_len = longest sentence (sizes the shared-memory ds buffer; <= 8192).
 * An empty sentence (0 rows) gets dgate, dv and dc 0. */
int edg_head_bwd(const void* h, int dtype, int64_t ldh, const int32_t* sent_ptr, int32_t B,
                 int32_t D, const float* gate, const float* v, const void* dist, int dist_i64,
                 const float* scores, const float* kl_b, const float* g_kl, const float* g_scores,
                 const float* g_pooled, const int32_t* arg, const void* g_xout, int64_t ldgx,
                 void* dh, int64_t lddh, float* dgate, float* dv, float* dc, int32_t max_len,
                 const int32_t* row_sent, int32_t N, edg_stream stream);

/* The gradient entering the GCN chain from scores / kl / the final max-pool (bert_amir5.py:639-648), already in the
 * aggregated form edg_gcn_layer (mode 1) and edg_wgrad consume, without reading h_L and without materialising dh_L:
 *   dh_L[t,:] = ds_t (gate o v_b) + [t == arg[b,:]] (gate o g_pooled_b),   ds_t = g_kl u_unit[t] (+ g_scores[t])
 *   du       = A^T dh_L         (bf16 [N, lddu]; mode 1 of edg_aggregate)
 *   dbias    = colsum(dh_L)     (fp32 [D], optional; fixed summation order)
 *   dgate    = g_kl v_b o sf_unit_b + g_pooled_b o hmax_b     (fp32 [B,D], optional: d loss / d gate_L)
 * u_unit [N] and sf_unit [B,D] come from edg_scores_kl_fwd, hmax / arg [B,D] from edg_gcn_layer (mode 0), tile_info /
 * n_tiles from edg_tile_plan.  g_kl: device scalar or NULL; g_scores [N], g_pooled / arg may be NULL.  D <= 320.
 * ws: edg_head_du_workspace(D) bytes when dbias is requested. */
size_t edg_head_du_workspace(int32_t D);
int edg_head_du(const float* u_unit, const float* g_kl, const float* g_scores, const float* gate, const float* v,
                const float* g_pooled, const int32_t* arg, const float* sf_unit, const float* hmax, int32_t N,
                int32_t B, int32_t D, const int32_t* row_ptr, const int32_t* col, const int32_t* sent_ptr,
                const int32_t* tile_info, const int32_t* n_tiles, void* du, int64_t lddu, float* dgate,
                float* dbias, void* ws, size_t ws_bytes, edg_stream stream);

/* x_out[i,:] = gate[b(i),:]*h[i,:]  (bert_amir5.py:639), only materialised when a
 * caller asks for the per-token output. */
int edg_gate_rows(const void* h, int dtype, int64_t ldh, const int32_t* sent_ptr, int32_t B,
                  int32_t D, const float* gate, void* out, int out_dtype, int64_t ldo,
                  edg_stream stream);

/* out[i,:] = act(gate[b(i),:]*h[i,:]), act = EDG_ACT_NONE or EDG_ACT_SIGMOID: the rows BertAmir54's
 * `fc = Sequential(Sigmoid, Linear)` (bert_amir5.py:464-465) scores, z = sigmoid(x_out).  Padding columns of `out`
 * are not written (allocate them zeroed). */
int edg_gate_rows_act(const void* h, int dtype, int64_t ldh, const int32_t* sent_ptr, int32_t B,
                      int32_t D, const float* gate, void* out, int out_dtype, int64_t ldo, int act,
                      edg_stream stream);

/* elementwise helper of the gate MLP backward: dz (+)= dy*y*(1-y) (nn.Sigmoid); writes the whole
 * [R, lddz] allocation (padding columns = 0). */
int edg_sigmoid_bwd(const void* y, int y_dtype, int64_t ldy, const void* dy, int dy_dtype,
                    int64_t lddy, int32_t R, int32_t C, void* dz, int dz_dtype, int64_t lddz,
                    int accumulate, edg_stream stream);

/* out[0] = scale * sum(in[0..n))   (deterministic; used for the batch means). */
int edg_sum_scaled(const float* in, int64_t n, float scale, float* out, edg_stream stream);

/* column sums of a [R,C] matrix -> fp32 out[C]; ws: edg_colsum_workspace bytes. */
size_t edg_colsum_workspace(int32_t R, int32_t C);
int edg_colsum(const void* x, int dtype, int64_t ldx, int32_t R, int32_t C, float* out,
               int accumulate, void* ws, size_t ws_bytes, edg_stream stream);

/* ------------------------------------------------------------------------- */
/* Neighbours of the path on the packed layout (SURVEY.md 8f)                  */
/* ------------------------------------------------------------------------- */

/* N1. Word-piece -> word averaging: `torch.bmm(transform, x)` of bert_amir5.py:600 (also bert_ed.py:50,
 * bertdm.py:166) with the transform of data_utils.py:438-451 (entries 1/l over the l contiguous word pieces of a
 * word) as a segment mean:  y[i] = sum_{j < seg_len[i]} fl32(1/seg_len[i]) * x[seg_start[i] + j].
 * x [P, ldx] packed word-piece rows ([CLS]/[SEP]/padding pieces simply belong to no segment), y [N, ldy]
 * packed word rows.  A word without pieces gives a zero row. */
int edg_segment_mean(const void* x, int dtype, int64_t ldx, const int32_t* seg_start, const int32_t* seg_len,
                     int32_t N, int32_t D, void* y, int y_dtype, int64_t ldy, edg_stream stream);
/* its adjoint: dx[seg_start[i] + j] = fl32(1/seg_len[i]) * dy[i]; every other row of dx [P, lddx] is zeroed. */
int edg_segment_mean_bwd(const void* dy, int dtype, int64_t lddy, const int32_t* seg_start, const int32_t* seg_len,
                         int32_t N, int32_t D, void* dx, int64_t lddx, int32_t P, edg_stream stream);

/* N4. BertDM's dynamic pooling (bertdm.py:116-140 masks, :174-185 pooling): pooled[b] = [max over tokens
 * t <= anchor | max over tokens anchor < t < n] of `x*mask + 1`, minus 1, the maximum running over all T_pad
 * padded positions as in the reference (masked positions contribute 0).  pooled fp32 [B, 2D], arg int32 [B, 2D]
 * = global row of the maximum, -1 where a masked zero won (no gradient).  T_pad = the batch's padded length
 * (max sentence length, bertdm.py:148). */
int edg_lr_pool_fwd(const void* h, int dtype, int64_t ldh, const int32_t* sent_ptr, const int32_t* anchor,
                    int32_t B, int32_t D, int32_t T_pad, float* pooled, int32_t* arg, edg_stream stream);
/* dh[arg[b,j], j mod D] += g[b,j] for arg >= 0  (dh is accumulated into). */
int edg_lr_pool_bwd(const float* g, const int32_t* arg, int32_t B, int32_t D, void* dh, int dtype, int64_t lddh,
                    edg_stream stream);

/* Gate dropout (bert_amir5.py:624-625: nn.Dropout on the gate broadcast to [B,T,D], so one keep/drop decision per
 * (token, column), shared by every use of that gate).  h * (gate * m / (1-p)) == (h * m / (1-p)) * gate, so the mask
 * is applied to the rows:  y[t,d] (+)= x[t,d] * keep(t,d) / (1-p)  and the kernels of the block run unchanged on y;
 * the backward pass applies the same call to the row gradient.  keep(t,d) = mix32(mix32(t*0x9E3779B1 + klo) ^
 * (d*0x85EBCA77 + khi)) >= floor(p * 2^32) with klo = lo32(seed) ^ (stream_id * 0xC2B2AE3D), khi = hi32(seed),
 * mix32 = the lowbias32 finaliser (x ^= x>>16; x *= 0x7feb352d; x ^= x>>15; x *= 0x846ca68b; x ^= x>>16).
 * seed: DEVICE int64 scalar (so a captured CUDA graph sees a new seed every replay).  x, y: same dtype. */
int edg_dropout_rows(const void* x, int dtype, int64_t ldx, void* y, int64_t ldy, int32_t N, int32_t D,
                     const int64_t* seed, int32_t stream_id, float p, int accumulate, edg_stream stream);

/* ------------------------------------------------------------------------- */
/* Optimiser step (train.py:239-243 trains with torch.optim.Adam)             */
/* ------------------------------------------------------------------------- */

/* One Adam step over n <= 32 fp32 tensors in one launch (torch.optim.Adam semantics: bias-corrected, eps added to
 * sqrt(v / bc2); weight_decay is the L2 form; no amsgrad):
 *   g = grad * grad_scale (+ weight_decay * p);  m = beta1 m + (1 - beta1) g;  v = beta2 v + (1 - beta2) g^2
 *   p -= lr / (1 - beta1^t) * m / (sqrt(v) / sqrt(1 - beta2^t) + eps)
 * param / grad / exp_avg / exp_avg_sq / step / numel are HOST arrays of length n (device pointers inside).  step[i]:
 * device fp32 scalar, the tensor's own step count t (on the device so that a captured step replays correctly; per tensor
 * as in torch, where a parameter without gradient does not advance); incremented by one before the update. */
int edg_adam_multi(int32_t n, void* const* param, const void* const* grad, void* const* exp_avg,
                   void* const* exp_avg_sq, void* const* step, const int64_t* numel, float lr, float beta1,
                   float beta2, float eps, float weight_decay, float grad_scale, edg_stream stream);

/* ------------------------------------------------------------------------- */
/* fp32-parity projection on the tensor cores (models/gcn.py:34, fp32 mode)   */
/* ------------------------------------------------------------------------- */

/* The tensor cores take no fp32 inputs, so the fp32 mode carries an fp32 matrix x as two fp16 matrices stored side by
 * side in one row, [ hi | lo ] with hi = fp16(x s), lo = fp16(x s - hi), s a power of two chosen from max|x| (device
 * scalar `amax`) so that max|x s| lies in [2^13, 2^14); each half is zero-padded to a multiple of 64 columns.  hi + lo
 * carries 22 significant bits of x; a product of two split matrices is three fp16 tensor-core products
 * (hi hi + hi lo + lo hi) with fp32 accumulation, scaled back by 1/(s_a s_b): error ~2^-21 per product, i.e. the
 * 1e-5 parity bound of the fp32 mode holds (tests/test_gpu_b_kernels.py).  Nothing here synchronises with the host. */

/* SMs (1..148, default 148) the persistent projection kernel behind edg_linear (bf16) may occupy; returns the previous
 * value.  Process-wide and not thread-safe: set it around the one launch that should leave room for a concurrent
 * collective (parallel.GradientAllReducer.bucket) and restore it. */
int edg_set_sm_budget(int32_t n);

/* elements (fp16) per row of the split form of a matrix with `cols` columns: 2 * round_up(cols, 64) */
int64_t edg_split_pitch(int32_t cols);

/* x fp32 [rows, cols] (pitch ldx, multiple of 4) -> out fp16 [rows, ldo] with ldo = edg_split_pitch(cols); amax: device
 * float[1], written with max|x| (the scale the consumers re-derive). */
int edg_split_f16(const float* x, int64_t ldx, int32_t rows, int32_t cols, void* out, int64_t ldo, float* amax,
                  edg_stream stream);

/* 1 when edg_linear_split covers the shape (the hi+lo weight slice must fit in shared memory next to two stages) */
int edg_linear_split_ok(int32_t K, int32_t Nout);

/* C fp32 [M, Nout] = act(A W^T + bias) from the split forms A2 [M, K], W2 [Nout, K] (same pitch lda == ldw ==
 * edg_split_pitch(K)) and their amax scalars.  Replaces edg_linear for fp32 operands (same bias / act / padding rules:
 * columns [Nout, ldc) of C are written as zeros). */
int edg_linear_split(const void* A2, int64_t lda, const float* amax_a, int32_t M, int32_t K, const void* W2, int64_t ldw,
                     const float* amax_w, int32_t Nout, const float* bias, int act, float* C, int64_t ldc,
                     edg_stream stream);

/* dW fp32 [K1, K2] = A^T B (+ dbias as in edg_wgrad: bias_of 1 = column sums of A, 2 = of B) from the split forms
 * A2 [R, K1], B2 [R, K2].  ws: edg_wgrad_split_workspace(R, K1, K2) bytes. */
size_t edg_wgrad_split_workspace(int32_t R, int32_t K1, int32_t K2);
int edg_wgrad_split(const void* A2, int64_t lda, const float* amax_a, int32_t K1, const void* B2, int64_t ldb,
                    const float* amax_b, int32_t K2, int32_t R, float* dW, int64_t lddw, float* dbias, int bias_of,
                    void* ws, size_t ws_bytes, edg_stream stream);

/* ------------------------------------------------------------------------- */
/* Classifier head and loss (bert_amir5.py:643 self.dense, train.py:121)      */
/* ------------------------------------------------------------------------- */

/* The classifier head and the collapsed-scores operands (bert_amir5.py:643-646, SURVEY A9) as ONE launch.  Per row b:
 *   pooled_b = g_b * p_b              (written to pooled [B, D] contiguous; when g == NULL pooled_b = p_b, nothing written)
 *   logits_b = W [a_b | pooled_b] + bias                  (W fp32 [C, 2D], bias [C] or NULL; logits [B, C] contiguous)
 *   va_b = logits_b^T fc_w[:, D:],  c_b = a_fc_b . va_b + logits_b . fc_b,  v_b = logits_b^T fc_w[:, :D]  (v [B, D] contiguous)
 * so that scores[b,t] = x_out[b,t,:] . v_b + c_b (edg_scores_kl_fwd).  a_fc is a, or sigmoid(a) for fc =
 * Sequential(Sigmoid, Linear).  All fp32, C <= 64.  Either head may be left out (not both):
 *   W == NULL (the logits come from a torch head): logits is an input; only v and c are written (a, p, g, pooled, bias
 *     unused);
 *   fc_w == NULL (a DenseHead on its own): only logits (and pooled when g is given) are written (a_fc, fc_b, v, c
 *     unused).
 * Each sum has the same order in every mode, so the combined launch gives the bits of the two composed. */
int edg_block_head_fwd(const float* a, int64_t lda, const float* a_fc, int64_t ldf, const float* p, int64_t ldp,
                       const float* g, int64_t ldg, const float* W, int64_t ldw, const float* bias, const float* fc_w,
                       int64_t ldfw, const float* fc_b, int32_t B, int32_t D, int32_t C, float* pooled, float* logits,
                       float* v, float* c, edg_stream stream);

/* Its input gradients as ONE launch.  With s = *scale (1 when NULL) and u_b = [s dv_b | s dc_b a_fc_b]:
 *   dlg_b = g_logits_b + fc_w u_b + s dc_b fc_b                                               (dlg [B, C] contiguous)
 *   da_b  = s dc_b (logits_b^T fc_w[:, D:]) (times a_fc (1 - a_fc) when fc_sigmoid) + dlg_b^T W[:, :D]
 *   dp_b  = dlg_b^T W[:, D:] + g_pooled_b                                          (da, dp [B, D] contiguous)
 * dv [B, D] / dc [B] (contiguous) are both NULL when the scores carry no gradient; g_logits [B, C] and g_pooled [B, D]
 * (contiguous) may be NULL.  logits [B, C] contiguous.  As in the forward, either head may be left out:
 *   W == NULL: dlg and da get the fc terms only; dp is not written (may be NULL);
 *   fc_w == NULL: dv and dc must be NULL; dlg = g_logits, da = dlg W[:, :D], dp = dlg W[:, D:] + g_pooled (logits,
 *     a_fc, fc_b unused).
 * The combined launch gives the bits of the fc-only launch followed by the dense-only one with g_logits = its dlg, the
 * two d a summed as da_dense + da_fc. */
int edg_block_head_bwd(const float* logits, const float* a, int64_t lda, const float* a_fc, int64_t ldf, int fc_sigmoid,
                       const float* W, int64_t ldw, const float* fc_w, int64_t ldfw, const float* fc_b, const float* dv,
                       const float* dc, const float* scale, const float* g_logits, const float* g_pooled, int32_t B,
                       int32_t D, int32_t C, float* dlg, float* da, float* dp, edg_stream stream);

/* The parameter gradients of the two: per-block partials in one launch, summed in block order by a second one.
 *   dv / dc given:  d_fc_w [C, 2D] = logits^T u,  d_fc_b [C] = logits^T (s dc)
 *   dlg given:      dW [C, 2D] = dlg^T [a | pooled],  dbias [C] = colsum(dlg)  (dbias may be NULL; logits may be NULL
 *                   when dv / dc are not given)
 * (all outputs contiguous, overwritten).  ws: edg_block_head_wgrad_workspace bytes. */
size_t edg_block_head_wgrad_workspace(int32_t B, int32_t D, int32_t C);
int edg_block_head_wgrad(const float* logits, const float* dlg, const float* a, int64_t lda, const float* a_fc,
                         int64_t ldf, const float* pooled, int64_t ldp, const float* dv, const float* dc,
                         const float* scale, int32_t B, int32_t D, int32_t C, float* dW, float* dbias, float* d_fc_w,
                         float* d_fc_b, void* ws, size_t ws_bytes, edg_stream stream);

/* nn.CrossEntropyLoss (mean reduction, ignore_index): out = device float[2] {mean loss over the rows whose target is not
 * ignore_index, number of such rows}; bad = device int[1], OR-ed with 1 when a target lies outside [0, C) (checked by the
 * caller when it chooses to: nothing here synchronises).  The backward writes
 * dlogits[b, c] = (softmax(logits_b)[c] - [c == target_b]) * (*gscale) / count (gscale NULL = 1), zero rows for ignored
 * targets; fwd_out is the forward's `out`.  ws: edg_cross_entropy_workspace(B) bytes of per-block partial sums whose last
 * 4 bytes are a ticket counter: zero before the first call, left zero by every call. */
size_t edg_cross_entropy_workspace(int32_t B);
int edg_cross_entropy_fwd(const float* logits, int64_t ldl, const int64_t* target, int32_t B, int32_t C,
                          int64_t ignore_index, float* out, int32_t* bad, void* ws, size_t ws_bytes, edg_stream stream);
int edg_cross_entropy_bwd(const float* logits, int64_t ldl, const int64_t* target, int32_t B, int32_t C,
                          int64_t ignore_index, const float* gscale, const float* fwd_out, float* dlogits, int64_t lddl,
                          edg_stream stream);

/* train.py:115-118: loss = t0 w0 + t1 w1 + t2 w2 on device scalars (CE + gate_weight xy + kl_weight kl; a NULL term
 * counts as zero), and its backward: out3[i] = (*g) w_i (g NULL = 1).  One launch each instead of four / six. */
int edg_loss_combine(const float* t0, const float* t1, const float* t2, float w0, float w1, float w2, float* out,
                     edg_stream stream);
int edg_loss_combine_bwd(const float* g, float w0, float w1, float w2, float* out3, edg_stream stream);

/* ---- Trigger pairs: every candidate trigger of a sentence from one pass of the GCN chain ----------------------------
 * The LitBank reader makes one example per (sentence, candidate trigger) pair; the GCN chain h_1 .. h_L depends on the
 * sentence only (its input x carries no trigger marker), so the sentence's rows are run once and only what depends on
 * the trigger runs per pair.  S sentences own rows [sent_ptr[s], sent_ptr[s+1]); the P pairs are grouped by sentence,
 * pairs of sentence s = [pair_ptr[s], pair_ptr[s+1]) (a sentence may have none); pair_sent[P] names each pair's
 * sentence, pair_start[P] = sent_ptr[pair_sent], anchor[P] is sentence-local.  Per-pair row data (distances, scores)
 * lives in the per-pair packed layout: pair p's copy of its sentence's n rows starts at pair_row_ptr[p] (P+1 entries).
 * Every sum over the pairs of a sentence runs in ascending pair order in one thread: results are deterministic.
 * The forward trigger gather is edg_trigger_gather with sent_ptr = pair_start and B = P. */

/* edg_tree_dist per pair: pair p walks sentence pair_sent[p] from anchor[p]; dist[pair_row_ptr[P]] is per-pair packed. */
int edg_tree_dist_pairs(const int32_t* row_ptr, const int32_t* col, const int32_t* sent_ptr, const int32_t* pair_sent,
                        const int32_t* pair_row_ptr, const int32_t* anchor, int32_t P, int32_t max_len, int32_t* dist,
                        edg_stream stream);
/* edg_scores_kl_fwd per pair over the sentence rows h [N, ldh]: gate, v fp32 [P,D], c fp32 [P] (NULL = 0), dist per-pair
 * packed; scores [pair_row_ptr[P]], kl_b [P]; optional dv_unit [P,D], dc_unit [P], u_unit [pair_row_ptr[P]],
 * sf_unit [P,D] as in edg_scores_kl_fwd with the mean taken over the P pairs (u_t = P_t (Q_t - kl_b) / P).
 * A pair whose sentence is empty gets kl_b 0 and zero unit outputs. */
int edg_scores_kl_pairs_fwd(const void* h, int dtype, int64_t ldh, const int32_t* sent_ptr, const int32_t* pair_sent,
                            const int32_t* pair_row_ptr, int32_t P, int32_t D, const float* gate, const float* v,
                            const float* c, const void* dist, int dist_i64, float* scores, float* kl_b, float* dv_unit,
                            float* dc_unit, float* u_unit, float* sf_unit, edg_stream stream);
/* Backward of the per-pair scores / kl and the final pool (pooled_p = gate_p * max_t h_t), same two-pass contract as
 * edg_head_bwd.  With ds_{p,t} = g_kl / P * P_{p,t} (Q_{p,t} - kl_b[p]) + g_scores[pair_row_ptr[p] + t]:
 *   first pass (dh = dgate = NULL): dv_p = gate_p * sum_t ds_{p,t} h_t, dc_p = sum_t ds_{p,t};
 *   full pass: dh [N, lddh] (compute dtype, every row written)
 *     dh_t = sum_{p of s} ds_{p,t} (gate_p * v_p) + [t = arg[s]] sum_{p of s} gate_p * g_pooled_p,
 *   dgate_p = v_p * sum_t ds_{p,t} h_t + g_pooled_p * h[arg[s]], and dv / dc when given.
 * arg int32 [S,D] = the sentence's global arg-max rows (-1 for an empty sentence), g_pooled fp32 [P,D] (NULL = 0).
 * ds_ws: fp32 workspace of pair_row_ptr[P] entries.  row_sent[N] (sentence of every row) is needed for dh.
 * With P = 0 the per-pair arrays may be NULL: dh (when given) is written as 0, nothing else is written. */
int edg_head_bwd_pairs(const void* h, int dtype, int64_t ldh, const int32_t* sent_ptr, int32_t S, const int32_t* row_sent,
                       int32_t N, const int32_t* pair_ptr,
                       const int32_t* pair_sent, const int32_t* pair_row_ptr, int32_t P, int32_t D, const float* gate,
                       const float* v, const void* dist, int dist_i64, const float* scores, const float* kl_b,
                       const float* g_kl, const float* g_scores, const float* g_pooled, const int32_t* arg, void* dh,
                       int64_t lddh, float* dgate, float* dv, float* dc, float* ds_ws, edg_stream stream);
/* edg_views_bwd_hmax per pair: gates / dgates [V,P,D], hmax [S,D] of the sentences;
 *   patch_val[s,d] = sum_{p of s} sum_v gates[v,p,d] dP_{v,p},  dgates[v,p,d] (+)= dP_{v,p} * hmax[s,d]
 * with dP_{v,p} = g_xy / P * sum_{v' != v} gates[v',p,d] * hmax[s,d].  A sentence without pairs gets patch_val 0. */
int edg_views_bwd_hmax_pairs(const float* hmax, const float* gates, const float* g_xy, int32_t V, int32_t S,
                             const int32_t* pair_ptr, int32_t P, int32_t D, float* patch_val, int64_t ldp, float* dgates,
                             int acc_view, edg_stream stream);
/* Gate dropout of the pairs (bert_amir5.py:624-625 on the expanded batch): pair p reads row t of its sentence under the
 * edg_dropout_rows mask of that row's copy, keep(seed, stream, pair_row_ptr[p] + t, column), so for one seed the pairs
 * apply exactly the masks the expanded batch applies; a kept element reads as T(h * 1/(1-p)) (rounded to the row dtype),
 * a dropped one as 0.  Streams: v for view v of h_1, L-1 for the final pool / scores of h_L.  seed: device int64 scalar,
 * p in [0, 1).  Masks are regenerated from the seed in both directions (nothing is stored per (pair, row)).
 *
 * Gated max-pool of the masked rows per pair, views v = 0..V-1 under streams stream0 + v (gates [V,P,D]): mmax [V,P,D]
 * = column maximum of the pair's masked rows, pooled = mmax * gates, arg = its first row (global sentence row; the
 * sentence's first row where the gate is 0).  A pair of an empty sentence gets pooled 0, arg -1, mmax 0; P = 0 does
 * nothing. */
int edg_pool_drop_pairs(const void* h, int dtype, int64_t ldh, const int32_t* sent_ptr, const int32_t* pair_sent,
                        const int32_t* pair_row_ptr, int32_t P, int32_t D, const float* gates, int32_t V,
                        const int64_t* seed, int32_t stream0, float p, float* pooled, int32_t* arg, float* mmax,
                        edg_stream stream);
/* edg_scores_kl_pairs_fwd on the masked rows of stream stream_id (same outputs, same empty-sentence and P = 0 rules). */
int edg_scores_kl_drop_pairs_fwd(const void* h, int dtype, int64_t ldh, const int32_t* sent_ptr, const int32_t* pair_sent,
                                 const int32_t* pair_row_ptr, int32_t P, int32_t D, const float* gate, const float* v,
                                 const float* c, const void* dist, int dist_i64, float* scores, float* kl_b,
                                 float* dv_unit, float* dc_unit, float* u_unit, float* sf_unit, const int64_t* seed,
                                 int32_t stream_id, float p, edg_stream stream);
/* edg_head_bwd_pairs on the masked rows of stream stream_id, with the final pool per pair: arg int32 [P,D] and mmax fp32
 * [P,D] from edg_pool_drop_pairs (dgate_p = v_p * sum_t ds_{p,t} m_{p,t} + g_pooled_p * mmax_p) and
 *   dh_t = sum_{p of s} keep_{p,t} / (1-p) * (ds_{p,t} gate_p v_p + [t = arg_p] gate_p g_pooled_p)
 * (every row written; 0 where the sentence has no pairs, so P = 0 gives dh = 0).  A pair of an empty sentence gets
 * dgate, dv and dc 0. */
int edg_head_bwd_drop_pairs(const void* h, int dtype, int64_t ldh, const int32_t* sent_ptr, int32_t S,
                            const int32_t* row_sent, int32_t N, const int32_t* pair_ptr, const int32_t* pair_sent,
                            const int32_t* pair_row_ptr, int32_t P, int32_t D, const float* gate, const float* v,
                            const void* dist, int dist_i64, const float* scores, const float* kl_b, const float* g_kl,
                            const float* g_scores, const float* g_pooled, const int32_t* arg, const float* mmax, void* dh,
                            int64_t lddh, float* dgate, float* dv, float* dc, float* ds_ws, const int64_t* seed,
                            int32_t stream_id, float p, edg_stream stream);
/* BertAmir54 on the pairs (bert_amir5.py:464-465 fc = Sequential(Sigmoid, Linear), applied at :538 before the scores
 * of :645-648): pair p scores the sigmoid of its gated rows, z_{p,t} = T(sigmoid(gate_p * h~_{p,t})) -- the value
 * edg_gate_rows_act stores, T the row dtype -- against v_p with a unit gate.  h~_{p,t} is row t of the pair's sentence
 * as stored (seed = NULL) or under the pair's mask of dropout stream stream_id (seed given; as edg_scores_kl_drop_pairs_fwd).
 * gate_p does not factor out of the sigmoid, so z is formed from each row as it is read; nothing is stored per
 * (pair, row).  Replaces the materialised z rows of the unpaired BertAmir54 path (edg_gate_rows_act + edg_scores_kl_fwd
 * with a unit gate) for a batch holding each sentence once.
 *
 * Forward: scores_{p,t} = sum_d z_{p,t,d} v_{p,d} + c_p, kl_b as edg_scores_kl_pairs_fwd, optional dv_unit [P,D] =
 * sum_t u_t z_{p,t} (no gate factor), dc_unit [P] = sum_t u_t.  Same empty-sentence, P = 0 and D rules. */
int edg_scores_kl_sig_pairs_fwd(const void* h, int dtype, int64_t ldh, const int32_t* sent_ptr, const int32_t* pair_sent,
                                const int32_t* pair_row_ptr, int32_t P, int32_t D, const float* gate, const float* v,
                                const float* c, const void* dist, int dist_i64, float* scores, float* kl_b,
                                float* dv_unit, float* dc_unit, const int64_t* seed, int32_t stream_id, float p,
                                edg_stream stream);
/* Its backward with the final pool, the two-pass contract of edg_head_bwd_pairs, ds_{p,t} as there:
 *   dc_p = sum_t ds_{p,t},  dv_p = sum_t ds_{p,t} z_{p,t},
 *   dgate_p = v_p * sum_t ds_{p,t} z (1 - z) h~_{p,t} + g_pooled_p * h[arg],
 *   dh_t = sum_{p of s} [keep_{p,t} / (1-p)] gate_p * (ds_{p,t} v_p z (1 - z)) + (arg-max term),
 * one thread per (row, 16-byte chunk) reading h_t once and the sentence's pairs in ascending order.  seed = NULL:
 * arg int32 [S,D] per sentence and the arg-max term of edg_head_bwd_pairs (mmax unused); seed given: arg / mmax [P,D]
 * per pair and the arg-max term of edg_head_bwd_drop_pairs.  Every row of dh is written (0 where the sentence has no
 * pairs; P = 0 gives dh = 0 and the per-pair arrays may be NULL). */
int edg_head_bwd_sig_pairs(const void* h, int dtype, int64_t ldh, const int32_t* sent_ptr, int32_t S,
                           const int32_t* row_sent, int32_t N, const int32_t* pair_ptr, const int32_t* pair_sent,
                           const int32_t* pair_row_ptr, int32_t P, int32_t D, const float* gate, const float* v,
                           const void* dist, int dist_i64, const float* scores, const float* kl_b, const float* g_kl,
                           const float* g_scores, const float* g_pooled, const int32_t* arg, const float* mmax, void* dh,
                           int64_t lddh, float* dgate, float* dv, float* dc, float* ds_ws, const int64_t* seed,
                           int32_t stream_id, float p, edg_stream stream);
/* Backward of the masked views (streams 0..V-1) and the diversity term from edg_pool_drop_pairs' pooled / mmax / arg
 * [V,P,D], with dP_{v,p} = g_xy / P * (sum_{v'} pooled_{v',p} - pooled_{v,p}):
 *   dgates (optional) [V,P,D]:  dgates[v,p] (+)= dP_{v,p} * mmax_{v,p}   (+= for v = acc_view)
 *   dh (optional, [N, lddh] compute dtype):  dh_t += sum_{p of s} sum_v [t = arg_{v,p}] keep_{v,p,t} / (1-p) gates_{v,p}
 *       dP_{v,p}, pairs then views in ascending order summed in fp32 and added once; rows no view routes to are not
 *       touched.  P = 0 does nothing. */
int edg_views_bwd_drop_pairs(const float* pooled, const float* mmax, const int32_t* arg, const float* gates,
                             const float* g_xy, int32_t V, const int32_t* sent_ptr, const int32_t* row_sent, int32_t N,
                             const int32_t* pair_ptr, const int32_t* pair_row_ptr, int32_t P, int32_t D,
                             const int64_t* seed, float p, void* dh, int dtype, int64_t lddh, float* dgates, int acc_view,
                             edg_stream stream);
/* edg_trigger_scatter_add per pair: dx[pair_start[p] + anchor[p]] += da[p] + sum_k extra[k][p], the pairs of a
 * sentence in ascending order (pairs may share a row). */
int edg_trigger_scatter_add_pairs(const float* da, const float* extra, int32_t n_extra, int32_t S, const int32_t* pair_ptr,
                                  int32_t P, int32_t D, const int32_t* pair_start, const int32_t* anchor, void* dx,
                                  int dtype, int64_t lddx, edg_stream stream);
/* N4 (edg_lr_pool_fwd) per pair over the sentence rows h [N, ldh]: pair p of sentence s with anchor a = anchor[p]
 * (sentence-local, inside the sentence) gets pooled[p] = [max over rows t <= a | max over rows a < t < n] of the
 * sentence, as edg_lr_pool_fwd gives p's copy of the sentence: the same T_pad rule for the left pool's masked zero, the
 * same (m + 1) - 1 rounding and the same first-index ties (a real 0 beats the left's masked 0; a right row must be
 * strictly positive), so values and arg are bit for bit the expanded batch's with arg = the global SENTENCE row.
 * pooled fp32 [P, 2D], arg int32 [P, 2D] (-1 where a masked zero won).  Pairs may come in any order within their
 * sentence and may share an anchor.  Each sentence's rows are read twice (an ascending and a descending pass), whatever
 * its pair count; a sentence of more than 512 rows or 2048 pairs is scanned once per pair instead. */
int edg_lr_pool_pairs_fwd(const void* h, int dtype, int64_t ldh, const int32_t* sent_ptr, const int32_t* pair_ptr,
                          const int32_t* anchor, int32_t S, int32_t P, int32_t D, int32_t T_pad, float* pooled,
                          int32_t* arg, edg_stream stream);
/* its adjoint: dh[t, j] = sum_{p of s} ([arg[p, j] = t] g[p, j] + [arg[p, D + j] = t] g[p, D + j]) for the rows t of
 * sentence s, pairs in ascending order, summed in one thread (fp64 for fp32 dh, fp32 for bf16 dh) and rounded once.
 * g fp32 [P, 2D].
 * Every row of every sentence is written (0 where nothing routes, sentences without pairs included), so dh needs no
 * clearing; P = 0 writes zeros (g and arg may then be NULL). */
int edg_lr_pool_pairs_bwd(const float* g, const int32_t* arg, const int32_t* sent_ptr, const int32_t* pair_ptr, int32_t S,
                          int32_t P, int32_t D, void* dh, int dtype, int64_t lddh, edg_stream stream);

#ifdef __cplusplus
}
#endif
#endif /* EDGCN_H_ */
