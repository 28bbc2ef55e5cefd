/* plnlp_b200.h -- C ABI of the B200 (sm_100a) kernels behind the PLNLP hot path.
 *
 * The reference (zhitao-wang/PLNLP) is pure Python and has no FFI of its own; the
 * "interface each entry point replaces" is therefore the third-party kernel call made
 * at a reference line.  Every entry point below cites that reference file:line.
 *
 * Conventions
 *  - plain `extern "C"`, raw DEVICE pointers + int64 sizes + a `cudaStream_t` passed as
 *    `void*`; no torch types, no exceptions, no allocation, no retained pointers.
 *  - the caller owns every buffer, including workspaces (sized with the documented
 *    formulas / the *_workspace_bytes helpers).
 *  - return value: 0 = ok; < 0 = invalid argument (PLNLP_E_*); > 0 = the cudaError_t of a
 *    failed launch.  Kernels are enqueued asynchronously on `stream`.
 *  - no CPU fallback and no other-arch dispatch: the library is built for sm_100a only.
 *  - all matrices are row-major with an explicit leading dimension in ELEMENTS.
 */
#ifndef PLNLP_B200_H
#define PLNLP_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PLNLP_ABI_VERSION 1

#define PLNLP_E_NULL       (-1)  /* required pointer is NULL            */
#define PLNLP_E_SIZE       (-2)  /* negative / inconsistent size         */
#define PLNLP_E_ALIGN      (-3)  /* pointer / leading dim not aligned    */
#define PLNLP_E_UNSUPPORTED (-4) /* valid but not implemented combination */
#define PLNLP_E_WORKSPACE  (-5)  /* workspace too small                  */
#define PLNLP_E_DEVICE     (-6)  /* current device is not sm_100         */

/* loss kinds: /root/reference/plnlp/loss.py:5-8, 11-14, 31-35 */
#define PLNLP_LOSS_AUC 0
#define PLNLP_LOSS_HINGE_AUC 1
#define PLNLP_LOSS_WEIGHTED_HINGE_AUC 2
/* the remaining objectives of --loss_func (loss.py:17-28, 38-62; SURVEY.md 8f rank 3) */
#define PLNLP_LOSS_WEIGHTED_AUC 3
#define PLNLP_LOSS_ADA_AUC 4
#define PLNLP_LOSS_ADA_HINGE_AUC 5
#define PLNLP_LOSS_LOG_RANK 6
#define PLNLP_LOSS_CE 7
#define PLNLP_LOSS_INFO_NCE 8

/* GEMM epilogue activations */
#define PLNLP_ACT_NONE 0
#define PLNLP_ACT_RELU 1        /* relu, then inverted dropout when drop_p > 0 (layer.py:21-22, 84-85) */
#define PLNLP_ACT_RELU_GRAD 2   /* C = acc * (aux > 0 ? 1/(1-drop_p) : 0): backward of the above       */

int plnlp_abi_version(void);
/* 0 when the CURRENT cuda device is compute capability 10.x, PLNLP_E_DEVICE otherwise. */
int plnlp_check_device(void);
/* number of kernels this library has launched since load (process-wide, for bench.py's
 * `gpu_launches`); reading it does not synchronise. */
int64_t plnlp_launch_count(void);

/* ------------------------------------------------------------------------------------
 * CSR row-gather SpMM (replaces torch_sparse.matmul under SAGEConv / GCNConv,
 * /root/reference/plnlp/layer.py:20,23, and its autograd backward which runs the same
 * kernel on the transposed structure, model.py:161).
 *
 *   out[r, :] = epi( (sum_{p in row r} val[p] * x[col[p], :]) / row_div[r] )
 *   epi(v) = dropout(relu(v + bias))   (each stage optional)
 *
 * The row set is described by a PLAN (built once per graph by the host, see
 * plnlp_b200/graph.py): work item i covers stored entries [item_ptr[i], item_ptr[i+1]) of row
 * item_row[i].  Rows no longer than the plan's chunk are one item (item_slot = -1, written
 * straight to `out`, accumulated strictly in CSR order -> bit-identical to the in-order CPU
 * loop).  Longer (hub) rows are split into several items that write fp32 partial sums to
 * partial[item_slot], combined in slot order by a second fixed-order pass (deterministic).
 *   fix_row[j] / fix_ptr[j..j+1] : split row j and its range of partial slots.
 * item_end (optional): explicit end offset of every item, for plans over a SUBSET of the rows (items are then
 * not contiguous); NULL = item i ends at item_ptr[i+1].  With a subset plan item_row holds the COMPACT output row.
 * Used for the forward of the LAST conv, whose output is only read at the endpoint rows of the edge batch
 * (model.py:152-156): ~10 % of citation2-shape's rows, ~25 % of the stored entries.
 * x_index (optional, one int32 per column of the adjacency): source j reads row x_index[j] of x; a negative
 * value is the caller's promise that this source row is all zeros -- it is skipped without being gathered
 * (the skipped terms are exact zeros and the surviving ones keep their order, so the result is unchanged).
 * Used for the backward of the last conv: the incoming gradient is non-zero only at the endpoint rows, either
 * as a compact [T, F] matrix (x_index = position in it) or as a full matrix (x_index[j] = j where row j is
 * non-zero, plnlp_row_nonzero_index_f32 builds that).
 * val == NULL: value-less adjacency.  row_div == NULL: no division (sum); SAGE mean passes
 * row_div[r] = max(row_nnz, 1) and gets the IEEE division upstream performs.
 * F: feature width; x/out leading dims in floats; x_rows: rows of x (every column index, or x_index value, is below
 * it -- the caller's promise; the kernels use it only to keep whole-vector copies of the last row inside the operand).
 * 16-byte vector loads are used when F, ldx, ldo are multiples of 4 and the bases are 16-byte aligned; otherwise 8- or
 * 4-byte.  fp32 operands of an even width <= 64 floats on a 16-byte aligned base run on the shared-memory staged
 * kernel (cp.async row copies, see plnlp_spmm_tune).
 * mask (optional, fp32 [rows, ldmask]): the forward activation Y = dropout(relu(.)) this product is the gradient of;
 * the epilogue then writes  Y[row, f] > 0 ? out * mask_scale : 0  -- the relu / dropout backward of the PREVIOUS layer
 * fused into the backward SpMM of the conv that consumed Y (layer.py:21-22), instead of a separate pass over [N, F].
 */
int plnlp_spmm_csr_f32(const int32_t* item_ptr, const int32_t* item_row, const int32_t* item_slot,
                       int64_t n_items, const int32_t* item_end, const int32_t* x_index,
                       const int32_t* col, const float* val,
                       const float* row_div, const float* bias, int relu, float drop_p, uint64_t seed,
                       const float* x, int64_t ldx, int64_t x_rows, float* out, int64_t ldo, int64_t F,
                       float* partial, const int32_t* fix_ptr, const int32_t* fix_row, int64_t n_fix,
                       const float* mask, int64_t ldmask, float mask_scale, void* stream);

/* Process-wide tuning of the SpMM gather kernels (A/B runs and the defaults plnlp_b200/_ops.py applies at load;
 * a negative / zero argument leaves that knob unchanged).  None of them changes a single output bit.
 *   prefetch_mode : 0 off; 1 = every lane asks the L2 for the row behind its column index as soon as the batch's
 *                   indices are known (prefetch.global.L2 per 128-byte line); 2 = the same with one
 *                   cp.async.bulk.prefetch.L2 per row; 3 = mode 2 for rows of 257..512 bytes, off otherwise (where it
 *                   was measured to pay).  All rows of a batch are then in flight at once instead of NB per warp.
 *   staged_mode   : 0 off; 1..12 = fp32 operands of an even width <= 64 floats run on the shared-memory staged kernel
 *                   (cp.async row copies; per warp a ring of 1: 16 rows x 4 stages, 2: 32 x 3, 3: 16 x 6, 4: 32 x 4,
 *                   5: 16 x 3, 6: 16 x 2, 7: 8 x 3, 8: 8 x 4, 9: 32 x 2, 10: 32 x 1, 11: 16 x 1; 12 = auto, the default:
 *                   32 x 1); staged_warps = warps per CTA (1..16).
 *   l2_fetch_bytes: cudaLimitMaxL2FetchGranularity (32 / 64 / 128) of the current device. */
int plnlp_spmm_tune(int prefetch_mode, int staged_mode, int staged_warps, int l2_fetch_bytes);

/* index[r] = r if any of x[r, 0..F) is non-zero (NaN counts as non-zero), else -1: an x_index of the SpMM. */
int plnlp_row_nonzero_index_f32(const float* x, int64_t ldx, int64_t rows, int64_t F, int32_t* index, void* stream);

/* The same SpMM on bf16 feature storage (the "bf16 path, stated separately" of BASELINE.json's north_star;
 * config 5 sweeps fp32 and bf16): x and out hold bf16 bit patterns, leading dims in ELEMENTS; every output
 * element is accumulated in fp32 in CSR order and rounded once (RN) at the store; val / row_div / bias and
 * the partial slots of split rows stay fp32.  Halves the gathered bytes: nnz*F*2 per launch.  16-byte loads
 * (8 features per lane) for F >= 256, 8-byte for F >= 128, 4-byte below, alignment permitting. */
int plnlp_spmm_csr_bf16(const int32_t* item_ptr, const int32_t* item_row, const int32_t* item_slot,
                        int64_t n_items, const int32_t* item_end, const int32_t* x_index,
                       const int32_t* col, const float* val,
                        const float* row_div, const float* bias, int relu, float drop_p, uint64_t seed,
                        const uint16_t* x, int64_t ldx, int64_t x_rows, uint16_t* out, int64_t ldo, int64_t F,
                        float* partial, const int32_t* fix_ptr, const int32_t* fix_row, int64_t n_fix,
                        const float* mask, int64_t ldmask, float mask_scale, void* stream);

/* ------------------------------------------------------------------------------------
 * Dense layers (replace torch.nn.Linear -> cuBLAS sgemm under SAGEConv.lin_l/lin_r,
 * GCNConv.lin, MLPPredictor.lins: layer.py:20,23,82-86, and their two backward GEMMs).
 *
 *   C = act( op(A) . op(B) + beta * C + bias )       op(A): M x K, op(B): K x N
 *   transa = 0: A[m*lda + k]     transa = 1: A[k*lda + m]
 *   transb = 0: B[k*ldb + n]     transb = 1: B[n*ldb + k]   (torch Linear weight layout)
 * split_k > 1 needs workspace of split_k*M*N floats; partials are reduced in split order
 * (deterministic).  aux (ldaux) is the forward activation for PLNLP_ACT_RELU_GRAD.
 * K = 0 gives act(beta * C + bias) and reads neither A nor B (either may be NULL).
 * plnlp_gemm_f32 is the exact-fp32 CUDA-core path (FFMA, fp32 accumulate).
 */
int plnlp_gemm_f32(int transa, int transb, int64_t M, int64_t N, int64_t K,
                   const float* A, int64_t lda, const float* B, int64_t ldb,
                   float* C, int64_t ldc, float beta, const float* bias, int act,
                   const float* aux, int64_t ldaux, float drop_p, uint64_t seed,
                   float* workspace, int64_t workspace_bytes, int split_k, void* stream);

/* Same contract on the 5th-generation tensor cores: tcgen05.mma kind::tf32, operands staged in
 * shared memory, fp32 accumulator in TMEM (csrc/gemm_tcgen05.cu).
 *   passes = 3: error-compensated 3xTF32 (A = Ah + Al, B = Bh + Bl; Ah.Bh + Ah.Bl + Al.Bh), ~1e-6
 *               relative to the fp32 result -- the parity path;
 *   passes = 1: plain TF32 (~1e-3 relative) -- the stated fast path. */
int plnlp_gemm_tf32(int passes, int transa, int transb, int64_t M, int64_t N, int64_t K,
                    const float* A, int64_t lda, const float* B, int64_t ldb,
                    float* C, int64_t ldc, float beta, const float* bias, int act,
                    const float* aux, int64_t ldaux, float drop_p, uint64_t seed,
                    float* workspace, int64_t workspace_bytes, int split_k, void* stream);

/* Same again with CTA pairs (tcgen05.mma.cta_group::2, csrc/gemm_tcgen05_2cta.cu): two SMs share one
 * 256 x 256 tile, each staging half of the B operand. */
int plnlp_gemm_tf32_2cta(int passes, int transa, int transb, int64_t M, int64_t N, int64_t K,
                         const float* A, int64_t lda, const float* B, int64_t ldb,
                         float* C, int64_t ldc, float beta, const float* bias, int act,
                         const float* aux, int64_t ldaux, float drop_p, uint64_t seed,
                         float* workspace, int64_t workspace_bytes, int split_k, void* stream);

/* TMA-fed persistent variant for the TALL-SKINNY dense layers of the full-graph encoder (csrc/gemm_tma.cu;
 * layer.py:20,23 at citation2 shape: 2.9 M x 200 x 178, 2.9 M x 50 x 200): A tiles arrive by cp.async.bulk.tensor
 * (128-byte swizzle) into a deep ring, the weight is split once per call into tf32 hi / lo copies in the caller's
 * workspace (plnlp_gemm_tf32_tma_workspace_bytes) and TMA-loaded as well, the TMEM accumulator is double buffered
 * so the epilogue of one tile overlaps the main loop of the next.  A is [M, K] row-major (lda % 4 == 0, 16-byte
 * aligned); transb = 1: B is [N, K] (y = x W^T), transb = 0: B is [K, N] (dX = dY W).  32 <= K, N <= 512, no split-k;
 * anything else returns PLNLP_E_UNSUPPORTED (-4) and the caller picks another kernel.  Same epilogue contract. */
int64_t plnlp_gemm_tf32_tma_workspace_bytes(int64_t N, int64_t K);
int plnlp_gemm_tf32_tma(int passes, int transb, int64_t M, int64_t N, int64_t K,
                        const float* A, int64_t lda, const float* B, int64_t ldb,
                        float* C, int64_t ldc, float beta, const float* bias, int act,
                        const float* aux, int64_t ldaux, float drop_p, uint64_t seed,
                        float* workspace, int64_t workspace_bytes, void* stream);

/* Weight gradients over a huge row count:  C[M, N] = A^T . B  with A [K, M] (lda) and B [K, N] (ldb) row-major, M, N <= 256
 * (dW = dY^T [A_hat x | 1] of the first encoder layer, layer.py:20,23 backward: 200 x 179 x 2 927 963).  TMA-fed,
 * persistent, tcgen05.mma on MN-major operands straight from the TMA boxes (nothing is transposed), hi / lo split by
 * convert warps, one accumulator per 1088 K-rows combined with RN adds, CTA partials added in CTA order
 * (deterministic).  lda, ldb multiples of 4, bases 16-byte aligned, N >= 8.  workspace: one [256][256] fp32 partial per SM. */
int64_t plnlp_gemm_tf32_tma_tn_workspace_bytes(void);
int plnlp_gemm_tf32_tma_tn(int passes, int64_t M, int64_t N, int64_t K, const float* A, int64_t lda,
                           const float* B, int64_t ldb, float* C, int64_t ldc, float* workspace,
                           int64_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------
 * Edge scoring (replaces h[edge[0]], h[edge[1]] advanced indexing + MLPPredictor /
 * DotPredictor, model.py:152-156,180 and layer.py:80-87,174-176).
 * `edges` is the reference's own int64 [P, 2] tensor (row p = (src, dst)).  h has n_rows rows;
 * a negative node index i addresses row n_rows + i, like the python indexing it replaces
 * (model.py:191-194 appends a mean row so that index -1 resolves).
 */
/* FUSED forward of the 2-layer MLP head over gathered endpoints (model.py:152-156 + layer.py:80-87):
 *   a0 = h[src_p] * h[dst_p]               gathered inside the GEMM's operand loader, never written to HBM
 *   a1 = dropout(relu(a0 @ W1^T + b1))     tcgen05 CTA-pair GEMM; stored to `a1` [P, N1] only if a1 != NULL
 *   score_part[q*score_ld + p] = a1[p, cols of partial q] . w2,   q in [0, 2*ceil(N1/256))
 * the caller adds the partials in index order plus the output bias.  passes as plnlp_gemm_tf32. */
int plnlp_edge_mlp_fwd_tf32(int passes, const float* h, int64_t ldh, int64_t n_rows, const int64_t* edges,
                            int64_t P, int64_t H, const float* W1, int64_t ldw, const float* b1, int64_t N1,
                            float drop_p, uint64_t seed, const float* w2, float* a1, int64_t lda1,
                            float* score_part, int64_t score_ld, void* stream);

/* Fused edge scoring, MLP head BACKWARD (model.py:161 through layer.py:80-87).  With a1 = dropout(relu(a0 W1^T + b1))
 * stored by plnlp_edge_mlp_fwd_tf32 and dscore = d loss / d score (plnlp_pair_loss_f32):
 *     dZ1 = (dscore (x) w2) . [a1 > 0] * drop_scale      formed inside the operand loaders, never written to HBM
 *     dA0 = dZ1 @ W1                    [P, H]           gradient of the Hadamard product (plnlp_edge_scatter_* next)
 *     dW1 = dZ1^T @ (h[src] * h[dst])   [N1, H]          the Hadamard product is re-gathered by the loader
 * Neither dZ1 nor the Hadamard product round-trips through HBM (before: 537 MB written and read twice each at the
 * ddi shape).  dw2 / db2 / db1 = colsum(dZ1) come from plnlp_mlp_out_bwd_f32 with dz = NULL.  H, N1 and the leading
 * dimensions must be multiples of 4, bases 16-byte aligned, N1 <= 1088.  dW1 is a split-k product over the P pairs:
 * workspace = plnlp_edge_mlp_bwd_workspace_bytes(P, H, N1, split_k) bytes, partials combined in split order. */
int64_t plnlp_edge_mlp_bwd_workspace_bytes(int64_t P, int64_t H, int64_t N1, int split_k);
int plnlp_edge_mlp_bwd_tf32(int passes, const float* h, int64_t ldh, int64_t n_rows, const int64_t* edges,
                            int64_t P, int64_t H, const float* W1, int64_t ldw, int64_t N1,
                            const float* a1, int64_t lda1, const float* dscore, const float* w2,
                            float drop_scale, float* dA0, int64_t ldda0, float* dW1, int64_t lddw1,
                            float* workspace, int64_t workspace_bytes, int split_k, void* stream);
/* out[p, :] = h[src_p, :] * h[dst_p, :] */
int plnlp_gather_hadamard_f32(const float* h, int64_t ldh, int64_t n_rows, const int64_t* edges, int64_t P, int64_t H,
                              float* out, int64_t ldo, void* stream);
/* Per-destination softmax over the stored entries of each CSR row and its backward: the attention weights of
 * torch_geometric.nn.TransformerConv under the reference's Transformer encoder (layer.py:57-63).
 *   alpha[e] = softmax over e in [rowptr[r], rowptr[r+1]) of scale * s[e]
 *   ds[e]    = scale * alpha[e] * (dalpha[e] - sum_{e' in row} alpha[e'] * dalpha[e'])
 * The per-entry scores s are <query_i, key_j> from plnlp_edge_dot_fwd_f32 over the entry list; the weighted
 * aggregation of the values is plnlp_spmm_csr_f32 with val = alpha. */
int plnlp_segment_softmax_fwd_f32(const int64_t* rowptr, int64_t n_rows, const float* s, float scale, float* alpha,
                                  void* stream);
int plnlp_segment_softmax_bwd_f32(const int64_t* rowptr, int64_t n_rows, const float* alpha, const float* dalpha,
                                  float scale, float* ds, void* stream);
/* Attention scores of a CSR row block against separate query and key tables: score[e] = <q[row(e)], k[col(e)]> for
 * every stored entry e, written in CSR entry order.  The block is walked through its SpMM work plan (item_ptr has
 * n_items + 1 offsets into col; item i holds the entries [item_ptr[i], item_ptr[i+1]) of row item_row[i]; graph.py
 * build_plan), so hub rows are split across warps.  q is [n_q, F] with leading dimension ldq, k is [n_k, F] with ldk.
 * Each score is bit-identical to plnlp_edge_dot_fwd_f32 over the pairs (row, n_q + col) of the stacked table [q; k].
 * Serves the row-partitioned TransformerConv (layer.py, _ops.BlockAttention): forward s = score(q, k) and backward
 * dalpha = score(g, v). */
int plnlp_attn_score_csr_f32(const int32_t* item_ptr, const int32_t* item_row, int64_t n_items, const int32_t* col,
                             const float* q, int64_t ldq, const float* k, int64_t ldk, int64_t F, float* score,
                             void* stream);

/* Plain endpoint gather out[p, :] = h[idx[p * idx_stride], :] (negative indices wrap) and its backward
 * grad_h[n, :] = sum_{t in segment n} g[entry[t], :] over a node-sorted entry list (seg_ptr has n_seg + 1
 * offsets, one segment per node, empty segments write zero rows; fixed summation order -> deterministic).
 * Replace x_i = h[edge[0]], x_j = h[edge[1]] (model.py:155-156) and autograd's index_put_(accumulate) for the
 * predictors that consume the two rows separately (MLPCatPredictor / MLPDotPredictor / MLPBilPredictor,
 * layer.py:90-164).  idx_stride = 2 reads one column of an int64 [P, 2] edge tensor in place. */
int plnlp_gather_rows_f32(const float* h, int64_t ldh, int64_t n_rows, const int64_t* idx, int64_t idx_stride,
                          int64_t P, int64_t H, float* out, int64_t ldo, void* stream);
int plnlp_row_scatter_sorted_f32(const float* g, int64_t ldg_in, int64_t H, const int64_t* seg_ptr,
                                 int64_t n_seg, const int64_t* entry, float* grad_h, int64_t ldg, void* stream);

/* score[p] = sum_d h[src_p, d] * h[dst_p, d]   (DotPredictor) */
int plnlp_edge_dot_fwd_f32(const float* h, int64_t ldh, int64_t n_rows, const int64_t* edges, int64_t P, int64_t H,
                           float* score, void* stream);
/* last MLP layer (out_channels = 1): score[p] = a[p, :] . w + b[0] */
int plnlp_mlp_out_fwd_f32(const float* a, int64_t lda, const float* w, const float* b, int64_t P,
                          int64_t H, float* score, void* stream);
/* backward of the above fused with the relu/dropout mask of `a`:
 *   dz[p, j] = dscore[p] * w[j] * (a[p, j] > 0 ? drop_scale : 0)     (mask_a != 0)
 *   dw[j] = sum_p dscore[p] * a[p, j];  db[0] = sum_p dscore[p]
 *   dzsum[j] = sum_p dz[p, j]   (optional: the bias gradient of the layer that produced `a`)
 * dz == NULL: dz is not written (the fused backward plnlp_edge_mlp_bwd_tf32 forms it in its loaders).
 * workspace: plnlp_mlp_out_bwd_workspace_bytes(P, H) bytes.  Deterministic. */
int64_t plnlp_mlp_out_bwd_workspace_bytes(int64_t P, int64_t H);
int plnlp_mlp_out_bwd_f32(const float* a, int64_t lda, const float* w, const float* dscore, int64_t P,
                          int64_t H, int mask_a, float drop_scale, float* dz, int64_t lddz, float* dw,
                          float* db, float* dzsum, void* workspace, int64_t workspace_bytes, void* stream);
/* Backward of the endpoint gather (replaces index_put_(accumulate=True), model.py:161).
 *   g[p, :] = da[p, :]            (MLP head; da = d loss / d hadamard)       or
 *   g[p, :] = dscore[p]           (DOT head; da == NULL)
 *   grad_h[src_p] += g[p] * h[dst_p];   grad_h[dst_p] += g[p] * h[src_p]
 * _atomic: red.global.add (order non-deterministic).  _sorted: one warp per node segment of
 * the node-sorted incidence list (entry = 2*p + side), fixed summation order; grad_h rows of
 * listed nodes are OVERWRITTEN.  seg_node == NULL: segment i is node i (n_seg <= n_rows, empty
 * segments write a zero row, so with n_seg == n_rows no zero fill is needed); otherwise the
 * caller zero-fills grad_h first. */
int plnlp_edge_scatter_atomic_f32(const float* h, int64_t ldh, int64_t n_rows, const int64_t* edges, int64_t P, int64_t H,
                                  const float* da, int64_t ldda, const float* dscore, float* grad_h,
                                  int64_t ldg, void* stream);
int plnlp_edge_scatter_sorted_f32(const float* h, int64_t ldh, int64_t n_rows, const int64_t* edges, int64_t P, int64_t H,
                                  const float* da, int64_t ldda, const float* dscore,
                                  const int64_t* seg_ptr, const int64_t* seg_node, int64_t n_seg,
                                  const int64_t* entry, float* grad_h, int64_t ldg, void* stream);

/* ------------------------------------------------------------------------------------
 * Pairwise losses + d loss / d score in one pass (replaces loss.py:5-8, 11-14, 31-35 and
 * their autograd mirror).  pos [B], neg [B, num_neg] (row i = negatives of positive i,
 * model.py:153), weight [B] (WeightedHingeAUC only).  loss[0] = SUM over pairs (not mean).
 * workspace: plnlp_pair_loss_workspace_bytes(B) bytes, contents arbitrary. Deterministic. */
int64_t plnlp_pair_loss_workspace_bytes(int64_t B);
int plnlp_pair_loss_f32(int kind, const float* pos, const float* neg, const float* weight, int64_t B,
                        int num_neg, float* loss, float* dpos, float* dneg, void* workspace,
                        int64_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------
 * Elementwise / reductions around the layers.
 */
/* dx = dy * (y > 0 ? scale : 0): backward of relu(+dropout) given the forward OUTPUT y
 * (layer.py:21-22, 25-26). */
int plnlp_relu_drop_bwd_f32(const float* y, int64_t ldy, const float* dy, int64_t lddy, float scale,
                            int64_t rows, int64_t cols, float* dx, int64_t lddx, void* stream);
/* out[c] = scale * sum_r x[r, c]  (bias gradients; mean row of h, model.py:193).
 * workspace: plnlp_colsum_workspace_bytes(rows, cols). Deterministic. */
int64_t plnlp_colsum_workspace_bytes(int64_t rows, int64_t cols);
int plnlp_colsum_f32(const float* x, int64_t ldx, int64_t rows, int64_t cols, float scale, float* out,
                     void* workspace, int64_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------
 * Negative samplers (replace negative_sample.py:6-20 and 31-43; both run on the HOST in
 * the reference).  Outputs use the reference layout: int64 [E, num_neg, 2].
 */
/* local: src = pos[e, 0] repeated, dst ~ U[0, num_nodes) from Philox4x32-10(seed). */
int plnlp_local_neg_sample(const int64_t* pos_edges, int64_t E, int64_t num_nodes, int num_neg,
                           uint64_t seed, int64_t* out, void* stream);
/* global, stage 1: draw n_cand candidate cells (r, c) ~ U[0,N)^2; a candidate is VALID when
 * r != c and r*N + c is not in the sorted id list `edge_ids` (n_edges entries; the existing
 * edges, id = edge_index[0]*N + edge_index[1]).  Valid candidates are inserted into an
 * open-addressing table (table_keys / table_first, `table_size` a power of two >= 2*n_cand,
 * pre-filled with 0xFF bytes) keeping, per distinct id, the SMALLEST candidate index
 * (deterministic).  cand_ids[i] = id or -1 when invalid. */
int plnlp_global_neg_candidates(const int64_t* edge_ids, int64_t n_edges, int64_t num_nodes,
                                int64_t n_cand, uint64_t seed, int64_t* cand_ids,
                                unsigned long long* table_keys, int* table_first, int64_t table_size,
                                void* stream);
/* stage 2: keep[i] = 1 iff candidate i is valid and is the first occurrence of its id. */
int plnlp_global_neg_keep(const int64_t* cand_ids, int64_t n_cand, const unsigned long long* table_keys,
                          const int* table_first, int64_t table_size, uint8_t* keep, void* stream);

/* ------------------------------------------------------------------------------------
 * Ranking metrics (replace ogb Evaluator._eval_hits / _eval_mrr on CPU tensors,
 * utils.py:49-56, 67-76).
 */
/* kth[0] = K-th largest element of neg[0..n) (1-based K <= n).  workspace >= 8192 bytes. */
int plnlp_kth_largest_f32(const float* neg, int64_t n, int64_t K, float* kth, void* workspace,
                          int64_t workspace_bytes, void* stream);
/* count[0] = #{ i : pos[i] > thresh[0] }  (strict, as ogb). */
int plnlp_count_greater_f32(const float* pos, int64_t n, const float* thresh,
                            unsigned long long* count, void* stream);
/* per row r of neg [S, K]: gt[r] = #{neg > pos[r]}, ge[r] = #{neg >= pos[r]}. */
int plnlp_mrr_counts_f32(const float* pos, const float* neg, int64_t ldn, int64_t S, int64_t K,
                         int32_t* gt, int32_t* ge, void* stream);

/* ------------------------------------------------------------------------------------
 * Link recommendation over all nodes (csrc/topk.cu; an extension, no reference call site): a score chunk
 * s [Q, N] holds row q = the predictor scores of (node[q], j) for every candidate j.
 */
/* Known-link filter: s[q*lds + col[e]] = -inf for e in [rowptr[node[q]], rowptr[node[q]+1]);
 * when exclude_self != 0, also s[q*lds + node[q]] = -inf.  Columns outside [0, N) are ignored.
 * rowptr == col == NULL: no known links (self only).  node[q] must be a row of the CSR (the caller's promise). */
int plnlp_score_mask_f32(float* s, int64_t lds, int64_t Q, int64_t N, const int64_t* node,
                         const int64_t* rowptr, const int32_t* col, int exclude_self, void* stream);

/* Per row q of s [Q, N] (row-major, lds >= N):
 *  - 0 < k <= 1024: the k largest finite entries, by score descending then column ascending
 *    -> ids [Q, k], scores [Q, k]; the tail is (-1, -inf) when fewer than k are finite.  -0 ties with +0.
 *  - target != NULL: gt[q] / ge[q] = #{j != target[q], s_j finite, s_j > / >= target_score[q]}.
 *    target_score is read by the caller BEFORE masking.
 * k == 0 with ids == NULL: rank counts only.  k > 1024 is PLNLP_E_UNSUPPORTED, N >= 2^31 PLNLP_E_SIZE.
 * One read of s.  Deterministic; integer outputs are exact.
 * workspace: plnlp_topk_rows_workspace_bytes(Q, N, k) bytes, 16-byte aligned. */
int64_t plnlp_topk_rows_workspace_bytes(int64_t Q, int64_t N, int64_t k);
int plnlp_topk_rows_f32(const float* s, int64_t lds, int64_t Q, int64_t N, int64_t k,
                        const int64_t* target, const float* target_score,
                        int64_t* ids, float* scores, int32_t* gt, int32_t* ge,
                        void* workspace, int64_t workspace_bytes, void* stream);

/* Column-offset forms for one shard of the candidates: s [Q, N] covers the global candidate ids [col0, col0 + N)
 * (0 <= col0, col0 + N < 2^31, else PLNLP_E_SIZE).  The mask reads col[] and node[q] as global ids (a known link c
 * lands at column c - col0); the select reports global ids col0 + j, breaks ties on them and compares target[q]
 * with them.  plnlp_score_mask_f32 / plnlp_topk_rows_f32 are these with col0 = 0. */
int plnlp_score_mask_cols_f32(float* s, int64_t lds, int64_t Q, int64_t N, int64_t col0, const int64_t* node,
                              const int64_t* rowptr, const int32_t* col, int exclude_self, void* stream);
int plnlp_topk_rows_cols_f32(const float* s, int64_t lds, int64_t Q, int64_t N, int64_t col0, int64_t k,
                             const int64_t* target, const float* target_score,
                             int64_t* ids, float* scores, int32_t* gt, int32_t* ge,
                             void* workspace, int64_t workspace_bytes, void* stream);
/* Candidate-set forms: s [Q, C] holds the candidates cand[0 .. C), strictly ascending global node ids (the caller's
 * promise).  The mask finds each known link and node[q] by binary search in cand and skips an id that is not there.
 * The select keeps its keys on the column, which orders as the ids do, and reports ids cand[j]; target[q] is a global
 * id, compared with the column it occupies (none when it is not in cand, and then every column counts).
 * cand == NULL in plnlp_topk_rows_cand_f32 is plnlp_topk_rows_cols_f32; with cand, col0 must be 0
 * (PLNLP_E_UNSUPPORTED).  Workspace as plnlp_topk_rows_cols_f32. */
int plnlp_score_mask_cand_f32(float* s, int64_t lds, int64_t Q, int64_t C, const int64_t* cand, const int64_t* node,
                              const int64_t* rowptr, const int32_t* col, int exclude_self, void* stream);
int plnlp_topk_rows_cand_f32(const float* s, int64_t lds, int64_t Q, int64_t N, int64_t col0, int64_t k,
                             const int64_t* target, const float* target_score,
                             int64_t* ids, float* scores, int32_t* gt, int32_t* ge,
                             void* workspace, int64_t workspace_bytes, const int64_t* cand, void* stream);
/* Cross-shard merge: ids_in / scores_in [R, Q, k_in] (rank-major: the all-gather of R per-shard [Q, k_in] results)
 * -> ids / scores [Q, k] (1 <= k <= 1024): per row the k best entries of the R lists by score descending then id
 * ascending, the tail (-1, -inf).  An entry with id < 0 or a non-finite score is dead.  Keys are rebuilt from
 * (score, global id), so the result does not depend on R or on how the candidates were split. */
int plnlp_topk_merge_f32(const int64_t* ids_in, const float* scores_in, int64_t R, int64_t Q, int64_t k_in,
                         int64_t k, int64_t* ids, float* scores, void* stream);

/* ------------------------------------------------------------------------------------
 * Random-walk augmentation (SURVEY.md 8f rank 1; replaces torch_cluster.random_walk and the pair /
 * weight assembly of main.py:228-233, 241-253).  rowptr / col: the reference's int64 CSR arrays.
 */
/* walk [n_walks, L+1]: walk[n,0] = start[n]; each step moves to col[rowptr[cur] + floor(u*deg)] (stays
 * put when deg == 0).  rand [n_walks, L] supplies the uniforms u in [0,1) (parity tests), or NULL:
 * Philox4x32-10(seed). */
int plnlp_random_walk(const int64_t* rowptr, const int64_t* col, const int64_t* start, int64_t n_walks,
                      int walk_length, const float* rand, uint64_t seed, int64_t* walk, void* stream);
/* pairs [L*n_walks, 2] (j-major: all walks for j = 0, then j = 1, ...) = (walk[n,0], walk[n,j+1]),
 * weight = 1/(j+1), keep = 0 for self pairs (main.py:244-253). */
int plnlp_walk_pairs(const int64_t* walk, int64_t n_walks, int walk_length, int64_t* pairs, float* weight,
                     uint8_t* keep, void* stream);

/* ------------------------------------------------------------------------------------
 * Graph construction (csrc/graph_build.cu): what main.py does once per run before the hot path -- ToSparseTensor
 * (main.py:81-83), to_symmetric (main.py:109-110), set_diag + D^-1/2 A D^-1/2 (plnlp/utils.py:83-89) -- with
 * bit-exact index arrays.  An entry is the key row * n_cols + col; sorts are stable radix sorts of (key, position)
 * pairs; counts that depend on the data come back through device counters the caller reads once.
 * ------------------------------------------------------------------------------------ */
int plnlp_graph_make_keys(const int64_t* row, const int64_t* col, int64_t n, int64_t n_cols, int both, int drop_diag,
                          int64_t* keys, int64_t* pos, void* stream);
int plnlp_graph_diag_keys(int64_t n_diag, int64_t n_cols, int64_t* keys, int64_t* pos, int64_t pos0, void* stream);
int64_t plnlp_graph_sort_workspace_bytes(int64_t n);
int plnlp_graph_sort_pairs(const int64_t* keys_in, const int64_t* pos_in, int64_t n, int64_t n_rows, int64_t n_cols,
                           int has_dead, int64_t* keys_out, int64_t* pos_out, void* workspace, int64_t workspace_bytes,
                           void* stream);
int64_t plnlp_graph_unique_workspace_bytes(int64_t n);
int plnlp_graph_unique(const int64_t* keys_in, int64_t n, int64_t* keys_out, int64_t* n_out, const int64_t* pos,
                       const float* val, int64_t n_src, float* val_out, void* workspace, int64_t workspace_bytes,
                       void* stream);
int plnlp_graph_keys_to_csr(const int64_t* keys, int64_t n, int64_t n_rows, int64_t n_cols, int64_t* rowptr,
                            int64_t* col, void* stream);
int plnlp_graph_sym_normalize(const int64_t* rowptr, const int64_t* col, const float* val_in, int64_t n_rows, float* dis,
                              float* val_out, void* stream);

/* Row-subset SpMM plan of the last conv (graph.py build_subset_plan; the rows a batch reads, model.py:152-156):
 * count kernel -> caller's inclusive prefix sums of n_it / multi / n_slot -> fill kernel.  One host read per plan. */
int plnlp_subset_plan_count(const int64_t* rowptr, const int64_t* rows, int64_t T, int chunk, int64_t* n_it,
                            int64_t* multi, int64_t* n_slot, int64_t* len, void* stream);
int plnlp_subset_plan_fill(const int64_t* rowptr, const int64_t* rows, int64_t T, int chunk, const int64_t* first,
                           const int64_t* fixi, const int64_t* slot, const int64_t* n_it, int32_t* item_ptr,
                           int32_t* item_end, int32_t* item_row, int32_t* item_slot, int32_t* fix_ptr,
                           int32_t* fix_row, float* row_cnt, void* stream);

/* ------------------------------------------------------------------------------------
 * Common-neighbour link heuristics (plnlp_b200/heuristics.py; csrc/heuristic.cu): CN, Adamic-Adar and Resource
 * Allocation, the non-learned baselines of the OGB link-prediction tables.  rowptr int64 [n + 1] / col int32 [nnz]:
 * a cleaned CSR (every row sorted, distinct, without its diagonal entry).  out[p] (fp64) = the sum over the common
 * neighbours w of rows edges[p, 0] and edges[p, 1] of weight[w] (fp64 [n]), or their count when weight is NULL.
 * edges int64 [P, 2] with ids in [-1, n); a pair with a negative id has no common neighbour.  Run-to-run
 * deterministic.
 * ------------------------------------------------------------------------------------ */
int plnlp_link_heuristic_f64(const int64_t* rowptr, const int32_t* col, int64_t n, int64_t nnz, const double* weight,
                             const int64_t* edges, int64_t P, double* out, void* stream);
/* Common-neighbour lists (plnlp_b200/heuristics.py common_neighbour_lists, the NCN predictor): col_out int32
 * [out_ptr[P]] receives the common neighbours of rows edges[p, 0] and edges[p, 1] of the same cleaned CSR at
 * col_out[out_ptr[p] .. out_ptr[p + 1]), in ascending id order.  out_ptr int64 [P + 1]: out_ptr[0] = 0 and
 * out_ptr[p + 1] - out_ptr[p] = the CN count plnlp_link_heuristic_f64 gives the pair.  Ids in [-1, n) as above. */
int plnlp_common_neighbour_list(const int64_t* rowptr, const int32_t* col, int64_t n, int64_t nnz,
                                const int64_t* edges, int64_t P, const int64_t* out_ptr, int32_t* col_out,
                                void* stream);
/* Heuristic recommendation over all nodes (plnlp_b200/heuristics.py recommend / rank_against_all): a chunk of Qc
 * query nodes against W candidate columns, the nodes [col0, col0 + W) or, with cand != NULL (strictly ascending
 * global ids, col0 must then be 0, else PLNLP_E_UNSUPPORTED), the nodes cand[0 .. W).
 * Mark: bitmap uint32 [Qc, ceil(W / 32)], zeroed by the caller; bit c of row q is set when column c's node j lies
 * in R(w) = {j : w in N(j)} for some w in N(nodes[q]) -- the nodes sharing a neighbour with the query.  rowptr / col:
 * the cleaned table N; rrowptr / rcol: its transpose R (same n); item_ptr int64 [Qc + 1]: item_ptr[0] = 0 and
 * item_ptr[q + 1] - item_ptr[q] = |N(nodes[q])|.  Every pointer but cand is required when Qc > 0 and W > 0 (a table
 * without entries marks nothing: skip the call).  The final bitmap does not depend on the order of the writes. */
int plnlp_two_hop_mark(const int64_t* rowptr, const int32_t* col, const int64_t* rrowptr, const int32_t* rcol,
                       int64_t n, const int64_t* nodes, const int64_t* item_ptr, int64_t Qc, int64_t col0, int64_t W,
                       const int64_t* cand, uint32_t* bitmap, void* stream);
/* Score: s [Qc, W] (row stride lds >= W), zeroed by the caller.  For every set bit c of row q, s[q, c] = the value
 * plnlp_link_heuristic_f64 gives the pair (nodes[q], column c's node) -- the same routine, bit for bit -- rounded to
 * fp32 once (_f32) or kept in fp64 (_f64).  Unmarked entries are not written. */
int plnlp_two_hop_score_f32(const int64_t* rowptr, const int32_t* col, int64_t n, int64_t nnz, const double* weight,
                            const int64_t* nodes, int64_t Qc, int64_t col0, int64_t W, const int64_t* cand,
                            const uint32_t* bitmap, float* s, int64_t lds, void* stream);
int plnlp_two_hop_score_f64(const int64_t* rowptr, const int32_t* col, int64_t n, int64_t nnz, const double* weight,
                            const int64_t* nodes, int64_t Qc, int64_t col0, int64_t W, const int64_t* cand,
                            const uint32_t* bitmap, double* s, int64_t lds, void* stream);

/* ------------------------------------------------------------------------------------
 * Path-based link scores (plnlp_b200/paths.py; csrc/propagate.cu): one hop of Katz or Personalized PageRank for a
 * block of B source columns, B in {32, 64, 128, 256}.  x [n, B] fp32, node-major, row stride ldx >= B; for every
 * output row j of [r0, r0 + rows):
 *   y[j - r0, c] = fp32(cm * s + (src[c] == j ? ba : 0)),  s = sum over the entries w of row j of weight[w] * x[w, c]
 * (weight fp64 [n], or 1 per entry when NULL), with cm / ba the fp64 values whose bit patterns are c_bits / b_bits.
 * Products, sums, the multiply and the add are fp64 rounded to nearest (no contraction); one rounding to fp32.
 * The rows are walked through an SpMM work plan over their entries (item_ptr [n_items + 1], item_row, item_slot,
 * fix_ptr / fix_row for the n_fix split rows, as plnlp_spmm_csr_f32); an item's entries are summed in order, a split
 * row's partials (partial fp64 [n_partial, B]) in item order, so every bit depends on the plan and the inputs only.
 * src int64 [B]: the source node of each column, -1 for a padding column.  Every x and weight must be >= 0.
 * live_in uint8 [n] or NULL: 0 promises an all-zero row of x, which is then not read (this changes no bit).
 * live_out uint8 [rows] or NULL: 1 where the output row has a non-zero entry, else 0.  y [rows, B], row stride
 * ldy >= B.  x, y, ldx and ldy aligned to min(B / 32, 4) floats (PLNLP_E_ALIGN).  Run-to-run deterministic.
 * ------------------------------------------------------------------------------------ */
int plnlp_propagate_f32(const int32_t* item_ptr, const int32_t* item_row, const int32_t* item_slot, int64_t n_items,
                        const int32_t* col, const int32_t* fix_ptr, const int32_t* fix_row, int64_t n_fix,
                        double* partial, const double* weight, const float* x, int64_t ldx, const int64_t* src,
                        int64_t B, uint64_t c_bits, uint64_t b_bits, const uint8_t* live_in, uint8_t* live_out,
                        int64_t r0, int64_t rows, float* y, int64_t ldy, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PLNLP_B200_H */
