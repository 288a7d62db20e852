/*
 * b200gnn.h — C ABI of the B200-native sparse message-passing engine.
 *
 * This is the drop-in boundary for the hot path of chaitjo/efficient-gnns
 * (SURVEY.md §8b).  The reference reaches its sparse arithmetic through
 * un-vendored Python/C++ dependencies (torch_sparse / torch_scatter / PyG);
 * each entry point below names the reference call site (file:line, relative
 * to /root/reference) whose arithmetic it replaces.
 *
 * Conventions
 *   - All pointers are DEVICE pointers unless the name ends in `_host`.
 *   - The library never allocates or frees: callers own every buffer,
 *     including workspaces (size helpers are provided).
 *   - Every call is asynchronous on `stream` (a cudaStream_t passed as void*),
 *     performs no host<->device synchronisation and is safe under CUDA-graph
 *     capture.
 *   - Return value: 0 on success, a negative B200GNN_ERR_* otherwise.
 *     b200gnn_last_cuda_error() gives the CUDA error string of the last
 *     B200GNN_ERR_CUDA on the calling thread.
 *   - Engine-side indices are int32 (the Python host narrows the reference's
 *     int64 once, with a range check); features are fp32 row-major with an
 *     explicit leading dimension (in elements).
 */
#ifndef B200GNN_H_
#define B200GNN_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200GNN_OK 0
#define B200GNN_ERR_BAD_ARG (-1)
#define B200GNN_ERR_UNSUPPORTED (-2)
#define B200GNN_ERR_CUDA (-3)

#define B200GNN_REDUCE_SUM 0
#define B200GNN_REDUCE_MEAN 1

#define B200GNN_ABI_VERSION 1

int b200gnn_abi_version(void);
const char* b200gnn_error_string(int code);
const char* b200gnn_last_cuda_error(void);
/* Number of kernel launches issued through this library by the calling
 * process since load / since the last reset (bench.py's gpu_launches). */
int64_t b200gnn_launch_count(void);
void b200gnn_reset_launch_count(void);

/* ------------------------------------------------------------------ *
 * CSR chunk plan: load balance for power-law graphs.  Chunk c is the run of
 * consecutive rows starting at the first row r with
 *     rowptr[r] + r*row_cost >= c*chunk_nnz ,
 * so each chunk (= one warp of the SpMM kernel) holds about chunk_nnz
 * non-zeros (+ row_cost per row, which also spreads empty rows).
 *   n_chunks = b200gnn_csr_chunk_count(...)   (host arithmetic only)
 *   chunk_rowptr: int32[n_chunks+1], chunk_rowptr[n_chunks] = n_rows
 * ------------------------------------------------------------------ */
int64_t b200gnn_csr_chunk_count(int64_t n_rows, int64_t nnz, int32_t chunk_nnz,
                                int32_t row_cost);
int b200gnn_csr_chunk_plan(const int32_t* rowptr, int64_t n_rows, int64_t nnz,
                           int32_t chunk_nnz, int32_t row_cost,
                           int32_t* chunk_rowptr, void* stream);

/* ------------------------------------------------------------------ *
 * CSR hub plan.  Rows whose degree exceeds `hub_threshold` are split into
 * segments of `seg_len` non-zeros processed by whole CTAs, so one hub node
 * (ARXIV-shape: degree ~2e4) cannot serialise a warp.  Built once per graph
 * and cached next to rowptr, like torch_sparse's SparseStorage caches
 * rowcount/colptr/csr2csc (used via arxiv_pyg/gnn.py:236-240).
 *   counts_out: int32[2] = {n_hub_rows, n_segments}
 *   hub_rows:   int32[n_hub]  ascending row ids
 *   hub_segptr: int32[n_hub+1] exclusive prefix of per-row segment counts
 * ------------------------------------------------------------------ */
int b200gnn_csr_hub_count(const int32_t* rowptr, int64_t n_rows,
                          int32_t hub_threshold, int32_t seg_len,
                          int32_t* counts_out, void* stream);
int b200gnn_csr_hub_fill(const int32_t* rowptr, int64_t n_rows,
                         int32_t hub_threshold, int32_t seg_len,
                         int32_t* hub_rows, int32_t* hub_segptr,
                         int64_t n_hub, void* stream);

/* ------------------------------------------------------------------ *
 * Row-segmented CSR SpMM  Y[i,:] = reduce_{e in row i} val[e] * X[col[e],:]
 * Replaces torch_sparse spmm_sum / spmm_mean reached from
 *   GCNConv  arxiv_pyg/gnn.py:47,52   (reduce=sum, weighted)
 *   SAGEConv arxiv_pyg/gnn.py:79,84   (reduce=mean, val==NULL)
 *   adj_t.matmul(x, reduce='mean')  mag_pyg/gnn.py:162
 * and their backward (the same kernel on the CSC view).
 *   val  : NULL => all ones.
 *   bias : NULL or float[K]; added after the reduction (GCNConv `out += bias`).
 *   stat_partial : NULL or float[b200gnn_spmm_stat_slots()][2][K]; every slot
 *          receives a deterministic partial column sum (slot,0,:) and sum of
 *          squares (slot,1,:) of the rows of Y it produced, for the
 *          BatchNorm1d that follows the conv (arxiv_pyg/gnn.py:48).
 *   chunk_rowptr/n_chunks : plan from b200gnn_csr_chunk_plan (required).
 *   hub_* : plan from b200gnn_csr_hub_*; n_hub==0 disables the split path
 *          (then hub_threshold must be >= the maximum degree or INT32_MAX).
 *   hub_workspace : float[n_seg][K] scratch for segment partials.
 * MEAN divides by max(degree,1); empty rows give 0 (+bias).
 * ------------------------------------------------------------------ */
int64_t b200gnn_spmm_stat_slots(int64_t n_chunks, int64_t n_hub);
/* Kernel selection for tuning / A-B measurement: 0 = automatic (cp.async-pipelined kernel for K in
 * {128,256,512}, multi-row kernel for K <= 64, register-staged kernel otherwise), 1 = always the
 * register-staged kernel. */
void b200gnn_spmm_set_variant(int variant);
int b200gnn_spmm_csr_f32(const int32_t* rowptr, const int32_t* col,
                         const float* val, const float* X, int64_t ldx,
                         float* Y, int64_t ldy, int64_t n_rows, int64_t n_src,
                         int64_t K, int reduce, const float* bias,
                         float* stat_partial, const int32_t* chunk_rowptr,
                         int64_t n_chunks, int32_t hub_threshold,
                         int32_t seg_len, const int32_t* hub_rows,
                         const int32_t* hub_segptr, int64_t n_hub,
                         int64_t n_seg, float* hub_workspace, void* stream);
/* The same product with the C->R layout exchange of the multi-GPU engine fused into the epilogue: output row i is stored to
 * Y_ptrs[q][(i - row_off[q]) * ldy_dst + col_dst ...] for the rank q that owns it (HOST arrays: `world` peer-mapped device
 * pointers, world+1 ascending row offsets).  Supported where the TMA kernels (K % 128 == 0) or the narrow kernel (K <= 64,
 * no fused statistics) run, else B200GNN_ERR_UNSUPPORTED. */
int b200gnn_spmm_csr_scatter_f32(const int32_t* rowptr, const int32_t* col, const float* val, const float* X,
                                 int64_t ldx, float* const* Y_ptrs, const int32_t* row_off, int32_t world,
                                 int64_t ldy_dst, int64_t col_dst, int64_t n_rows, int64_t n_src, int64_t K,
                                 int reduce, const float* bias, const int32_t* chunk_rowptr, int64_t n_chunks,
                                 int32_t hub_threshold, int32_t seg_len, const int32_t* hub_rows,
                                 const int32_t* hub_segptr, int64_t n_hub, int64_t n_seg,
                                 float* hub_workspace, void* stream);

/* ------------------------------------------------------------------ *
 * Dense row-major [n_rows,K] passes between the aggregations of a layer:
 * BatchNorm1d(train) -> ReLU -> dropout (arxiv_pyg/gnn.py:48-50) and their
 * backward.  K % 4 == 0, K <= 1024, 16-byte aligned, contiguous (ld == K).
 * All reductions go through `partial[slots][2][K]` scratch with
 * slots = b200gnn_rows_slots(n_rows) (one CTA per slot, fixed order =>
 * deterministic).
 * ------------------------------------------------------------------ */
int64_t b200gnn_rows_slots(int64_t n_rows);
/* partial[s][0][:] = column sums, partial[s][1][:] = column sums of squares */
int b200gnn_col_stats_f32(const float* Y, int64_t n_rows, int64_t K,
                          float* partial, int64_t slots, void* stream);
/* out[K] = column sums of Y (bias gradient of the last conv) */
int b200gnn_col_sum_f32(const float* Y, int64_t n_rows, int64_t K, float* out,
                        float* partial, int64_t slots, void* stream);
/* partials (from the SpMM epilogue or col_stats) -> batch mean / invstd and the
 * fused affine  scale = gamma*invstd, shift = beta - mean*scale ; running
 * statistics updated like nn.BatchNorm1d (momentum, unbiased variance) unless
 * running_mean/running_var are NULL. */
int b200gnn_bn_finalize_f32(const float* partial, int64_t slots, int64_t K,
                            int64_t n_rows, const float* gamma,
                            const float* beta, float eps, float momentum,
                            float* running_mean, float* running_var,
                            float* mean_out, float* invstd_out,
                            float* scale_out, float* shift_out, void* stream);
/* out = dropout_p(relu(Y*scale + shift)); scale/shift NULL => identity affine;
 * relu: 0/1.  The keep-mask is a pure function of (seed, effective offset,
 * element index) (Philox4x32-10) with
 *     effective offset = offset + (step_dev ? *step_dev * step_mul : 0),
 * step_dev being a device int32 (e.g. the Adam step counter) so a captured
 * CUDA graph draws a fresh mask on every replay;
 * row_offset: global index of row 0 of Y (node-parallel shards draw the mask
 * of their own rows of the global matrix; 0 on a single GPU);
 * b200gnn_dropout_mask_u8 materialises the mask of a given effective offset.
 * Uniforms: when p*65536 is integral (the reference's p = 0.5) eight 16-bit
 * uniforms per Philox block, keep iff u16 >= p*65536 (exact); otherwise four
 * 24-bit uniforms per block, keep iff u >= p. */
int b200gnn_affine_relu_dropout_f32(const float* Y, float* out, int64_t n_rows,
                                    int64_t K, const float* scale,
                                    const float* shift, int relu, float p,
                                    uint64_t seed, uint64_t offset,
                                    const int32_t* step_dev, uint64_t step_mul,
                                    uint64_t row_offset, void* stream);
/* Block form (node-parallel engine, SURVEY.md §8e "identical dropout masks by global node id"): local row r is node
 * rowmap[r] (or r + row_offset when rowmap is NULL), local columns are [col_offset, col_offset + K) of a
 * K_global-wide matrix; every keep decision equals the one the full-matrix call takes for that (node, feature). */
int b200gnn_affine_relu_dropout_mapped_f32(const float* Y, float* out, int64_t n_rows, int64_t K,
                                           const float* scale, const float* shift, int relu, float p,
                                           uint64_t seed, uint64_t offset, const int32_t* step_dev,
                                           uint64_t step_mul, const int32_t* rowmap, uint64_t row_offset,
                                           int64_t K_global, int64_t col_offset, void* stream);
/* ... with the C->R layout exchange fused: every output row is ALSO stored to the R-layout buffer of the rank owning the node:
 * dst_ptrs[q] + (r - row_off[q]) * ld_dst + col_offset (HOST arrays of `world` peer-mapped device pointers / world+1 offsets). */
int b200gnn_affine_relu_dropout_scatter_f32(const float* Y, float* out, int64_t n_rows, int64_t K,
                                            const float* scale, const float* shift, int relu, float p,
                                            uint64_t seed, uint64_t offset, const int32_t* step_dev,
                                            uint64_t step_mul, const int32_t* rowmap, uint64_t row_offset,
                                            int64_t K_global, int64_t col_offset, float* const* dst_ptrs,
                                            const int32_t* row_off, int32_t world, int64_t ld_dst, void* stream);
int b200gnn_dropout_mask_u8(uint8_t* mask, int64_t n_rows, int64_t K, float p,
                            uint64_t seed, uint64_t offset, void* stream);
/* Backward of out = dropout_p(relu(Y)) (no normalisation, the R-GCN hidden layers, mag_pyg/gnn.py:134-135):
 * dY = dOut * [out > 0] / (1-p).  dY may alias dOut. */
int b200gnn_relu_dropout_bwd_f32(const float* dOut, const float* Xout, int64_t n_rows, int64_t K, float p, float* dY,
                                 void* stream);
/* The same with an upstream gradient added before the ReLU/dropout backward: the reference's ``model.out_feat`` is the last
 * hidden activation after ReLU and dropout (mag_pyg/gnn.py:133-136), so a loss on it joins the gradient coming back from
 * the logits layer there.  dY[i, c] = (dOut[i, c] + (c < K_extra ? dExtra[i * ld_extra + c] : 0)) * [Xout[i, c] > 0] / (1-p),
 * added, then scaled: bit-identical to b200gnn_relu_dropout_bwd_f32 on dOut + dExtra zero-padded to K columns.  dOut, Xout,
 * dY: [n_rows, K] (K a multiple of 4, 16-byte aligned); dExtra: [n_rows, K_extra] with row pitch ld_extra, no alignment
 * needed, 0 <= K_extra <= K.  dY may alias dOut. */
int b200gnn_relu_dropout_bwd_add_f32(const float* dOut, const float* dExtra, int64_t ld_extra, int64_t K_extra,
                                     const float* Xout, int64_t n_rows, int64_t K, float p, float* dY, void* stream);
/* Backward of out = dropout_p(relu(BN_train(Y))): given dOut, out (for the
 * mask: out>0 <=> kept and active), Y and the saved batch mean/invstd, writes
 * dY, dgamma[K], dbeta[K] and (if non-NULL) dbias[K] = column sums of dY.
 * coef: float[3*K] scratch.  dY must not alias dOut. */
int b200gnn_bn_act_bwd_f32(const float* dOut, const float* Xout, const float* Y,
                           const float* mean, const float* invstd,
                           const float* gamma, int64_t n_rows, int64_t K,
                           float p, float* dY, float* dgamma, float* dbeta,
                           float* dbias, float* partial, int64_t slots,
                           float* coef, void* stream);
/* The same backward in two phases, for node-parallel runs that all-reduce the
 * column sums between them: reduce -> partial[slots][2][K];  apply consumes
 * `sums[sum_slots][2][K]` (the local partials, or ONE slot of cross-rank sums)
 * with n_norm = global row count. */
int b200gnn_bn_act_bwd_reduce_f32(const float* dOut, const float* Xout,
                                  const float* Y, const float* mean,
                                  const float* invstd, int64_t n_rows,
                                  int64_t K, float p, float* partial,
                                  int64_t slots, void* stream);
int b200gnn_bn_act_bwd_apply_f32(const float* dOut, const float* Xout,
                                 const float* Y, const float* mean,
                                 const float* invstd, const float* gamma,
                                 const float* sums, int64_t sum_slots,
                                 int64_t n_norm, int64_t n_rows, int64_t K,
                                 float p, float* dY, float* dgamma,
                                 float* dbeta, float* dbias, float* partial,
                                 int64_t slots, float* coef, void* stream);
/* Xout == NULL in b200gnn_bn_act_bwd_apply_f32: dOut already holds
 * dz = dOut * [Xout > 0] / (1-p), as stored by b200gnn_gemm_tf32x3_bnbwd_f32
 * (whose partial buffer is then `sums`); dY may alias dOut. */
/* out[K2] = sum over slots of partial[slot][K2] (K2 = 2*K for statistics) */
int b200gnn_partial_reduce_f32(const float* partial, int64_t slots, int64_t K2,
                               float* out, void* stream);
/* torch.optim.Adam (defaults: no amsgrad, no weight decay) over flat buffers;
 * *step (device int32) is the number of steps already taken and is incremented
 * (arxiv_pyg/gnn.py:192-193, 308-315). */
int b200gnn_adam_step_f32(float* params, const float* grads, float* exp_avg,
                          float* exp_avg_sq, int64_t n, float lr, float beta1,
                          float beta2, float eps, int32_t* step, void* stream);

/* ------------------------------------------------------------------ *
 * Row-wise classification / logit-KD loss with its gradient in one pass.
 *   kd_criterion(logits[train_idx], labels[train_idx], teacher[train_idx],
 *                alpha, T)                  arxiv_pyg/criterion.py:8-21
 *   F.cross_entropy(out, labels)            arxiv_pyg/gnn.py:112  (teacher_logits == NULL)
 * logits / teacher_logits / dlogits are FULL [N,C] matrices (leading dims ld/ldt/ldd);
 * train_idx (int64[n_train], NULL => rows 0..n_train-1) selects the rows, labels is the
 * full int64[N] vector.  dlogits rows in train_idx receive d loss / d logits; the caller
 * zeroes the other rows.  loss_out[3] = {loss, loss_cls, loss_kd}.
 * n_norm: row count the means are taken over (0 => n_train; node-parallel
 * shards pass the GLOBAL number of training rows and sum loss_out across ranks).
 * partial: float[2*b200gnn_kd_partials(n_train)] scratch.  C <= 1024 (ogbn-mag: 349).
 * ------------------------------------------------------------------ */
int64_t b200gnn_kd_partials(int64_t n_train);
int b200gnn_kd_loss_fwd_bwd_f32(const float* logits, int64_t ld,
                                const int64_t* train_idx, int64_t n_train,
                                const int64_t* labels,
                                const float* teacher_logits, int64_t ldt,
                                int64_t C, float alpha, float T,
                                int64_t n_norm, float* dlogits, int64_t ldd,
                                float* loss_out, float* partial, void* stream);

/* ------------------------------------------------------------------ *
 * fp32-faithful dense GEMM on tcgen05 tensor cores (3xTF32 split, fp32
 * accumulation in TMEM):   C[M,N] = A[M,K] * B[N,K]^T (+ bias[N])
 * Replaces the fp32 cuBLAS contractions behind GCNConv's `x @ weight`,
 * nn.Linear and their input gradients (arxiv_pyg/gnn.py:47,52,79,84 via PyG).
 *   A    : fp32, row-major, split into tf32 hi/lo on the fly inside the kernel.
 *   B_hi, B_lo : the [N,K] operand pre-split by b200gnn_split_tf32_f32
 *          (weights are tiny; `transpose` lets [K,N] storage feed it).
 * lda/ldb multiples of 4 floats, 16-byte aligned bases (TMA); any M, N, K.
 * Dropped terms are O(2^-22) relative, i.e. within the 1e-5 parity budget.
 * ------------------------------------------------------------------ */
int b200gnn_split_tf32_f32(const float* W, int64_t rows, int64_t cols,
                           int transpose, float* hi, float* lo, void* stream);
int b200gnn_gemm_tf32x3_f32(const float* A, int64_t lda, const float* B_hi,
                            const float* B_lo, int64_t ldb, float* C,
                            int64_t ldc, int64_t M, int64_t N, int64_t K,
                            const float* bias, void* stream);
/* C += A · B^T (accumulating epilogue; same operands as above, no bias). */
int b200gnn_gemm_tf32x3_acc_f32(const float* A, int64_t lda, const float* B_hi, const float* B_lo,
                                int64_t ldb, float* C, int64_t ldc, int64_t M, int64_t N, int64_t K,
                                void* stream);
/* Grouped form over row ranges (the per-node-type weights of an R-GCN layer, mag_pyg/gnn.py:54-65), one launch:
 *   C[row0_g + m, :N] (+)= A[row0_g + m, :K_g] * B_g[N, K_g]^T (+ bias_g[N])   for m < rows_g, every group g.
 * A (pitch lda) and C (pitch ldc) are shared; each group brings its own pre-split B pair (pitch ldb), K_g (a multiple
 * of 4, <= lda) and optional bias.  Groups must not overlap in C.  rows_g = 0 is a no-op; K_g = 0 stores the bias alone
 * (zero without one), or leaves C unchanged when accumulating.  At most 16 groups.  Each group's tiles do the arithmetic
 * of b200gnn_gemm_tf32x3_f32 / _acc_f32 on that group, bit for bit. */
typedef struct b200gnn_gemm_group {
  const float* B_hi;
  const float* B_lo;
  int64_t ldb;
  const float* bias;
  int64_t row0, rows, K;
} b200gnn_gemm_group;
int b200gnn_gemm_tf32x3_grouped_f32(const float* A, int64_t lda, float* C, int64_t ldc, int64_t N,
                                    const b200gnn_gemm_group* groups, int32_t n_groups, int accumulate, void* stream);
/* Row passes fused into the GEMM epilogue (SURVEY §8 f1; the reference runs conv -> BatchNorm1d -> ReLU -> dropout as
 * separate full-matrix ops, arxiv_pyg/gnn.py:47-50, and autograd walks them again backwards).  Each epilogue warp keeps
 * running column sums over the tiles of its CTA and stores them once: partial[slots][2][N], slots >=
 * b200gnn_gemm_stat_slots(M, N), fixed summation order (deterministic).  N a multiple of 32, 48 < N <= 256, ldc % 4 == 0.
 *   _stats_f32 : C = A·B^T + bias (accumulate: C += A·B^T, no bias — SAGEConv's lin_l(mean) + lin_r(x)) and partial = per-slot (sum C, sum C^2) over rows — the BatchNorm batch statistics of C,
 *                input of b200gnn_bn_finalize_f32 (replaces the b200gnn_col_stats_f32 sweep).
 *   _bnbwd_f32 : the input-gradient GEMM of the layer BEHIND a BatchNorm->ReLU->dropout block with pass 1 of that block's
 *                backward in the epilogue: dOut = A·B^T (+ C if accumulate); dz = dOut * [Xout > 0] / (1-p) is what is STORED
 *                to C, partial = per-slot (sum dz, sum dz*xhat), xhat = (Y-mean)*invstd (replaces
 *                b200gnn_bn_act_bwd_reduce_f32; follow with b200gnn_bn_act_bwd_apply_f32(dOut = C, Xout = NULL, sums =
 *                partial)).  Xout, Y: [M, ldc] like C. */
int64_t b200gnn_gemm_stat_slots(int64_t M, int64_t N);
/* A/B knob for measurements: 0 automatic (Xout / Y of _bnbwd_f32 staged through TMA when N % 128 == 0), 2 = always the
 * register path. */
void b200gnn_gemm_set_bnbwd_variant(int v);
int b200gnn_gemm_tf32x3_stats_f32(const float* A, int64_t lda, const float* B_hi, const float* B_lo, int64_t ldb,
                                  float* C, int64_t ldc, int64_t M, int64_t N, int64_t K, const float* bias,
                                  int accumulate, float* partial, int64_t slots, void* stream);
int b200gnn_gemm_tf32x3_bnbwd_f32(const float* A, int64_t lda, const float* B_hi, const float* B_lo, int64_t ldb,
                                  float* C, int64_t ldc, int64_t M, int64_t N, int64_t K, int accumulate,
                                  const float* Xout, const float* Y, const float* mean, const float* invstd, float p_drop,
                                  float* partial, int64_t slots, void* stream);
/* Same GEMM with the R->C layout exchange of the multi-GPU engine fused into the epilogue: output columns
 * [q*kc, (q+1)*kc), kc = N/world (a multiple of 32), are stored to C_ptrs[q][(row_off + m)*kc + ...] — C_ptrs is a HOST array
 * of `world` device pointers (the ranks' [N_nodes, kc] buffers, peer-mapped), so the tile results cross NVLink as they are
 * produced and no separate exchange kernel runs (the caller follows with b200gnn_peer_barrier). */
int b200gnn_gemm_tf32x3_scatter_f32(const float* A, int64_t lda, const float* B_hi, const float* B_lo,
                                    int64_t ldb, float* const* C_ptrs, int32_t world, int64_t row_off,
                                    int64_t M, int64_t N, int64_t K, const float* bias, void* stream);
/* ... and the row all-gather of a narrow result fused the same way: the whole [M, N] tile block is stored to EVERY
 * C_ptrs[q] (row pitch ldc) at rows row_off + m. */
int b200gnn_gemm_tf32x3_bcast_f32(const float* A, int64_t lda, const float* B_hi, const float* B_lo,
                                  int64_t ldb, float* const* C_ptrs, int32_t world, int64_t row_off, int64_t ldc,
                                  int64_t M, int64_t N, int64_t K, const float* bias, void* stream);

/* Weight gradient  dW[Kin,Nout] = X[Nn,Kin]^T * G[Nn,Nout]  (GCNConv weight.grad / nn.Linear weight.grad^T),
 * split-K over the node index on tcgen05 (3xTF32), partials reduced in fixed order.
 * Kin in {128,256}, Nout a multiple of 4 up to 256 (else B200GNN_ERR_UNSUPPORTED: caller keeps the library GEMM).
 * workspace: float[b200gnn_wgrad_workspace_floats(Kin,Nout)]. */
int64_t b200gnn_wgrad_workspace_floats(int64_t Kin, int64_t Nout);
int b200gnn_gemm_wgrad_tf32x3_f32(const float* X, int64_t ldx, const float* G,
                                  int64_t ldg, float* dW, int64_t Nn,
                                  int64_t Kin, int64_t Nout, float* workspace,
                                  void* stream);
/* A/B knob for measurements: 0 automatic (separate correction accumulators / drains against the accumulator's
 * round-towards-zero), 1 drains only, 2 one accumulation chain per CTA (round-1 behaviour, 1e-5-level gradient error). */
void b200gnn_wgrad_set_mode(int mode);

/* ------------------------------------------------------------------ *
 * Feature-distillation criteria (arxiv_pyg/criterion.py): row / pair passes.
 * The S x S contractions (G-CRD logits, GSP Gram matrices) run on
 * b200gnn_gemm_tf32x3_f32; these kernels are the passes around them.
 * ------------------------------------------------------------------ */
/* F.normalize(x, p=2, dim=-1) * scale  (fitnet :30-31, gpw :68-69, nce :139-140); norm_out[n] = ||x|| */
int b200gnn_row_normalize_fwd_f32(const float* x, int64_t n, int64_t F, float eps,
                                  float scale, float* out, float* norm_out,
                                  void* stream);
int b200gnn_row_normalize_bwd_f32(const float* out, const float* norm,
                                  const float* d_out, int64_t n, int64_t F,
                                  float eps, float scale, float* d_x,
                                  int accumulate, void* stream);
/* scratch sizes for the deterministic scalar reductions below */
int64_t b200gnn_reduce_slots(int64_t n);
/* F.mse_loss(a, b): loss_out[0]; d_a (nullable) = grad_weight * 2 (a-b) / n; partial: float[b200gnn_reduce_slots(n)] */
int b200gnn_mse_fwd_bwd_f32(const float* a, const float* b, int64_t n,
                            float grad_weight, float* d_a, float* loss_out,
                            float* partial, void* stream);
/* F.binary_cross_entropy_with_logits(z, target) over n elements (ppi_pyg/criterion.py:11; target_is_logits != 0:
 * target = sigmoid(target), the teacher term of :13).  d_z (nullable) = grad_weight * (sigmoid(z) - t) / n */
int b200gnn_bce_logits_fwd_bwd_f32(const float* z, const float* target,
                                   int target_is_logits, int64_t n,
                                   float grad_weight, float* d_z, float* loss_out,
                                   float* partial, void* stream);
/* feat.pow(2).sum(-1)  (at_criterion :44-45) and its backward */
int b200gnn_row_sqnorm_f32(const float* x, int64_t n, int64_t F, float* out, void* stream);
int b200gnn_row_sqnorm_bwd_f32(const float* x, const float* d_out, int64_t n,
                               int64_t F, float* d_x, void* stream);
/* G-CRD / InfoNCE (nce_criterion :142-146) over logits Z[S,S] (already / tau):
 * loss_out[0] = mean_i(logsumexp_j Z_ij - Z_ii); Z is overwritten by d loss / d Z.  partial: float[S]. */
int b200gnn_nce_rows_f32(float* Z, int64_t S, float* loss_out, float* partial, void* stream);
/* The same pass on a ROW CHUNK of the logits (rows [row_offset, row_offset+n_rows), row pitch ldz >= S): the S x S
 * matrix of criterion.py:142-146 is never materialised — the caller streams L2-sized chunks GEMM -> this pass -> the two
 * backward GEMMs; b200gnn_nce_finish_f32 reduces partial[S] to the loss. */
int b200gnn_nce_rows_chunk_f32(float* Z, int64_t ldz, int64_t n_rows, int64_t S, int64_t row_offset,
                               float* partial, void* stream);
int b200gnn_nce_finish_f32(const float* partial, int64_t S, float* loss_out, void* stream);
int b200gnn_transpose_f32(const float* in, int64_t rows, int64_t cols, float* out, void* stream);
/* GSP (gpw_criterion :66-86): Gs/Gt = Gram matrices of the sampled student/teacher rows; kernel 0 cosine,
 * 1 poly, 2 l2, 3 rbf (ns/nt = row squared norms for 2,3).  loss_out[0] = mse(sim_s, sim_t); Gs is overwritten by
 * d loss / d Gs; rowcoef[S] (kernels 2,3) = sum_j d loss / d ns_i.  partial: float[S]. */
int b200gnn_gsp_pair_f32(float* Gs, const float* Gt, const float* ns, const float* nt,
                         int64_t S, int kernel, float* rowcoef, float* loss_out,
                         float* partial, void* stream);
/* y[i,:] += alpha * coef[i] * x[i,:] */
int b200gnn_row_axpy_f32(const float* x, const float* coef, int64_t n, int64_t F,
                         float alpha, float* y, void* stream);

/* ------------------------------------------------------------------ *
 * LSP (lpw_criterion, arxiv_pyg/criterion.py:95-126) on an edge list sorted by
 * destination (src/dst int32[E], rowptr int32[n_seg+1] over dst).
 * kernel: 0 cosine, 1 poly, 2 l2, 3 rbf.  criterion: 0 kld, 1 mse.
 *   edge_sim     : sim[e] = k(feat[src[e]], feat[dst[e]])
 *   lsp_segment  : PyG softmax per dst segment for student and teacher sims,
 *                  loss_out[0] = the reference's loss_lpw, g[e] = d loss / d sim_s[e]
 *   edge_sim_bwd : dfeat += chain rule of g through k (atomic row adds; dfeat pre-zeroed by the caller)
 * ------------------------------------------------------------------ */
int b200gnn_edge_sim_f32(const float* feat, int64_t F, const int32_t* src,
                         const int32_t* dst, int64_t E, int kernel, float* sim,
                         void* stream);
int64_t b200gnn_lsp_partials(int64_t n_seg);
int b200gnn_lsp_segment_f32(const float* sim_s, const float* sim_t,
                            const int32_t* rowptr, int64_t n_seg, int64_t E,
                            int criterion, float* g, float* loss_out,
                            float* partial, void* stream);
int b200gnn_edge_sim_bwd_f32(const float* feat, int64_t F, const int32_t* src,
                             const int32_t* dst, int64_t E, int kernel,
                             const float* sim, const float* g, float* dfeat,
                             void* stream);
/* Deterministic LSP backward: d feat = C · feat with the (2E + n_nodes)-entry matrix C whose CSR structure
 * (comb_rowptr, and per edge / per node the entry positions pos_dst, pos_src, diag_pos) the caller builds once per
 * edge list: entry pos_dst[e] sits in row dst[e] at column src[e], pos_src[e] in row src[e] at column dst[e],
 * diag_pos[i] at (i, i).  This call fills val[2E + n_nodes] (selfc is scratch of the same size); the product itself
 * is b200gnn_spmm_csr_f32 — fixed summation order, no atomics (criterion.py:95-126 backward). */
int b200gnn_lsp_bwd_values_f32(const float* feat, int64_t F, const int32_t* src, const int32_t* dst,
                               int64_t E, int kernel, const float* sim, const float* g,
                               const int32_t* pos_dst, const int32_t* pos_src,
                               const int32_t* comb_rowptr, const int32_t* diag_pos, int64_t n_nodes,
                               float* val, float* selfc, void* stream);

/* ------------------------------------------------------------------ *
 * Graph attention (BASELINE config 4): per-destination edge softmax and
 * multi-head weighted aggregation, CSR rows = destinations, col = sources.
 *   DGL GATConv.forward   arxiv_dgl/models.py:196-217  (softmax_eps = 0)
 *   PyG GATConv           ppi_pyg/gnn.py:27-31          (softmax_eps = 1e-16)
 *   gat_edge_softmax : a[e,h] = softmax_e( leaky_relu(el[col[e],h] + er[row,h]) )   er NULL => el only
 *   gat_aggregate    : out[r, h*D+d] = sum_e a[eidx ? eidx[e] : e, h] * ft[col[e], h*D+d]
 *                      (forward on the CSR; d ft on the transposed CSR with eidx = csr2csc)
 *   gat_bwd_rows     : given d out, writes dpre[e,h] = d loss / d (el+er)[e,h] and der[r,h]
 *   segment_sum_heads: out[r,h] = sum_e vals[eidx[e],h]  (d el over the transposed CSR)
 * H <= 16.  chunk_rowptr / hub_rows / hub_segptr: the plans of b200gnn_csr_chunk_plan / b200gnn_csr_hub_fill
 * (rows above hub_threshold are split into seg_len-edge segments, as in b200gnn_spmm_csr_f32).
 * hub_workspace: n_seg*H*D floats for gat_aggregate, n_seg*H floats for gat_bwd_rows (unused when n_hub == 0).
 * Teacher-training knobs (arxiv_dgl/models.py:206-214): edge_keep [nnz] uint8 (NULL = keep all) — dropped edges get
 * a = 0 and leave the softmax (edge_drop); attn_scale [nnz,H] (NULL = none) = keep/(1-p) of the attention dropout:
 * the caller aggregates with a*attn_scale and gat_bwd_rows chains d a = d(a*attn_scale) * attn_scale.
 * ------------------------------------------------------------------ */
int b200gnn_gat_edge_softmax_f32(const int32_t* rowptr, const int32_t* col,
                                 const float* el, const float* er, int64_t n_rows,
                                 int64_t H, float negative_slope, float softmax_eps,
                                 float* a, const uint8_t* edge_keep, void* stream);
int b200gnn_gat_aggregate_f32(const int32_t* rowptr, const int32_t* col,
                              const int32_t* eidx, const float* a, const float* ft,
                              int64_t ldf, float* out, int64_t ldo, int64_t n_rows,
                              int64_t H, int64_t D, const int32_t* chunk_rowptr,
                              int64_t n_chunks, int32_t hub_threshold, int32_t seg_len,
                              const int32_t* hub_rows, const int32_t* hub_segptr,
                              int64_t n_hub, int64_t n_seg, float* hub_workspace,
                              void* stream);
int b200gnn_gat_bwd_rows_f32(const int32_t* rowptr, const int32_t* col, const float* a,
                             const float* ft, int64_t ldf, const float* dout,
                             int64_t ldd, const float* el, const float* er,
                             int64_t n_rows, int64_t H, int64_t D,
                             float negative_slope, float* dpre, float* der,
                             const int32_t* chunk_rowptr, int64_t n_chunks,
                             int32_t hub_threshold, int32_t seg_len,
                             const int32_t* hub_rows, const int32_t* hub_segptr,
                             int64_t n_hub, int64_t n_seg, float* hub_workspace,
                             const float* attn_scale, void* stream);
int b200gnn_segment_sum_heads_f32(const int32_t* rowptr, const int32_t* eidx,
                                  const float* vals, int64_t n_rows, int64_t H,
                                  float* out, void* stream);

/* ------------------------------------------------------------------
 * Peer-memory exchange of the node-parallel engine (SURVEY.md §8e; no reference counterpart: the reference is
 * single-GPU, arxiv_pyg/scripts/run_gcn.sh:24-28).  One process per GPU; each rank allocates an exchange arena,
 * publishes its CUDA IPC handle (64 opaque bytes, exchanged by the host side, e.g. torch.distributed) and maps the
 * peers' arenas.  Exchange steps are kernels that store directly into the consumers' arenas over NVLink, then a
 * flag barrier:
 *   b200gnn_peer_copy2d_f32 : n <= 16 strided block copies in one launch, dst_j[r, 0:width] = src_j[r, 0:width]
 *                             (width % 4 == 0; 16-byte aligned bases and pitches); dst_j may be peer memory
 *   b200gnn_peer_barrier    : peer_flags[q] = rank q's flag array (16 uint64 slots, zero-initialised, inside its
 *                             arena) as mapped in THIS process (host array of `world` device pointers); stores
 *                             epoch+1 into slot [rank] of every rank's array with release semantics at system
 *                             scope, waits until its own slots all reached it, then bumps *epoch (device counter,
 *                             so the call is CUDA-graph replayable).  A peer that never arrives sets *error = 1
 *                             after ~2^27 polls instead of hanging the device.
 * ------------------------------------------------------------------ */
typedef struct b200gnn_copy2d {
  float* dst;
  const float* src;
  int64_t ld_dst; /* floats */
  int64_t ld_src; /* floats */
  int64_t rows;
} b200gnn_copy2d;
int b200gnn_arena_alloc(int64_t bytes, void** out);
int b200gnn_arena_free(void* ptr);
int b200gnn_ipc_get_handle(const void* dev_ptr, void* handle64);
int b200gnn_ipc_open_handle(const void* handle64, void** out);
int b200gnn_ipc_close_handle(void* ptr);
int b200gnn_peer_copy2d_f32(const b200gnn_copy2d* copies, int32_t n, int64_t width, void* stream);
int b200gnn_peer_barrier(uint64_t* const* peer_flags, int32_t rank, int32_t world,
                         uint64_t* epoch, int32_t* error, void* stream);
/* copy2d + barrier in ONE launch: the CTA that finishes last (ticket: device uint32, zero-initialised, re-armed by the
 * kernel) runs the flag barrier, so the kernel ends when every rank's blocks have been exchanged. */
int b200gnn_peer_exchange_f32(const b200gnn_copy2d* copies, int32_t n, int64_t width,
                              uint64_t* const* peer_flags, int32_t rank, int32_t world, uint64_t* epoch,
                              int32_t* error, uint32_t* ticket, void* stream);

/* ------------------------------------------------------------------
 * Heterogeneous input assembly — RGCN.group_input, mag_pyg/gnn.py:111-124 (called from RGCN.forward :126-129):
 *   out[i, :] = tables[node_type[i]][local_idx[i], :]     (tables[t] NULL or type out of range => zero row)
 * node_type / local_idx are the int64 tensors of group_hetero_graph; tables / table_rows are HOST arrays of
 * n_tables <= 16 device pointers / row counts.  An index outside its table sets *error_flag (device int32) to 1.
 * typed_scatter is the backward: d_tables[t][j, :] = sum over nodes i with (node_type, local_idx) == (t, j) of
 * d_out[i, :], written (not accumulated: untouched rows keep what the caller put there, normally zeros) for the
 * tables whose pointer is non-NULL.  `order` = the node ids sorted by (node_type, local_idx) (stable): runs of equal
 * keys are added in that order by one warp => deterministic, no atomics.
 * ------------------------------------------------------------------ */
int b200gnn_typed_gather_f32(const float* const* tables, const int64_t* table_rows, int32_t n_tables,
                             const int64_t* node_type, const int64_t* local_idx, int64_t n, int64_t F,
                             float* out, int64_t ldo, int32_t* error_flag, void* stream);
int b200gnn_typed_scatter_f32(const float* d_out, int64_t ldd, const int64_t* node_type,
                              const int64_t* local_idx, const int64_t* order, int64_t n, int64_t F,
                              float* const* d_tables, const int64_t* table_rows, int32_t n_tables,
                              void* stream);

/* ------------------------------------------------------------------
 * Graph ingestion on the device (SURVEY.md §8 f2) — the integer half of the data path, bit-exact:
 *   b200gnn_graph_argsort_i64  : perm = stable argsort of key = major*minor_size + minor.  ToSparseTensor
 *                                (arxiv_pyg/gnn.py:236-237: major = edge_index[1], minor = edge_index[0]), an unsorted
 *                                SparseTensor(row=, col=) (mag_pyg/gnn.py:151) and csr2csc (major = col, minor = row).
 *   b200gnn_graph_coalesce_i64 : COO -> row-sorted duplicate-free COO + rowptr (to_symmetric's coalesce,
 *                                arxiv_pyg/gnn.py:240).  out_row/out_col/src_out hold n entries, the first *nnz_out
 *                                (device int64) are valid; src_out (nullable) = input index of each kept entry.
 * Hand-written stable LSD radix sort (8-bit digits, only the digits the key range needs) + flags/scan/compaction +
 * binary-search row pointers.  workspace: b200gnn_graph_sort_workspace_bytes(n) bytes, 256-byte aligned.
 * n < 2^31; major_size*minor_size < 2^64.
 * ------------------------------------------------------------------ */
int64_t b200gnn_graph_sort_workspace_bytes(int64_t n);
int b200gnn_graph_argsort_i64(const int64_t* major, const int64_t* minor, int64_t n, int64_t major_size,
                              int64_t minor_size, int32_t* perm_out, void* workspace, void* stream);
int b200gnn_graph_coalesce_i64(const int64_t* row, const int64_t* col, int64_t n, int64_t n_rows,
                               int64_t n_cols, int64_t* out_row, int64_t* out_col, int32_t* src_out,
                               int64_t* rowptr_out, int64_t* nnz_out, void* workspace, void* stream);

/* ------------------------------------------------------------------
 * Mini-batch sampling on the device (SURVEY §8 f4) — replaces the CPU workers of
 * torch_geometric.data.GraphSAINTRandomWalkSampler as the reference drives it (mag_pyg/gnn.py:361-366: roots uniform
 * over the nodes, torch_sparse.random_walk of walk_length steps, SparseTensor.saint_subgraph of the visited nodes).
 *   random_walk: out[w][0] = start[w]; step s of walker w moves to col[rowptr[v] + (r * deg >> 32)], r = word (s % 4) of
 *     Philox4x32-10(seed, offset, w * ceil(L/4) + s / 4); a node without out-edges holds the walker.  out: [n_walks, L+1].
 *   saint_subgraph: induced subgraph of the sorted unique node set `nodes` over CSR, CSR order kept.  count -> per selected
 *     row the number of kept edges (and fills node_map, an int32 [n_nodes] workspace that holds -1 on entry); the caller
 *     prefix-sums the counts into out_ptr; fill -> local row / local col / parent edge id (eid[j], or j when eid is NULL).
 * ------------------------------------------------------------------ */
int b200gnn_random_walk_i64(const int32_t* rowptr, const int32_t* col, int64_t n_nodes, const int64_t* start,
                            int64_t n_walks, int32_t walk_length, uint64_t seed, uint64_t offset, int64_t* out,
                            void* stream);
int b200gnn_saint_subgraph_count_i64(const int32_t* rowptr, const int32_t* col, const int64_t* nodes, int64_t n_sel,
                                     int32_t* node_map, int64_t* counts, void* stream);
int b200gnn_saint_subgraph_fill_i64(const int32_t* rowptr, const int32_t* col, const int64_t* eid, const int64_t* nodes,
                                    int64_t n_sel, const int32_t* node_map, const int64_t* out_ptr, int64_t* out_row,
                                    int64_t* out_col, int64_t* out_eid, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* B200GNN_H_ */
