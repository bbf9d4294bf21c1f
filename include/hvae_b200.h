/* hvae_b200 -- C ABI of the B200-native HybridVAE hot path (libhvae_b200.so).
 *
 * The reference (Aymane-Nouhail/Recommendation-System) has no FFI layer: its hot path is stock PyTorch
 * (ATen) calls issued from src/ml/model.py, src/ml/train.py and src/ml/evaluate.py.  Each entry point
 * below replaces the ATen call sequence cited next to it (paths relative to the reference root).  The
 * Python package `hvae_b200` binds these symbols with ctypes and exposes them as torch custom ops
 * (`torch.ops.hvae_b200.*`); see INTEGRATION.md for the binding a reference maintainer would add.
 *
 * Conventions: every pointer is a DEVICE pointer unless stated otherwise; the caller owns all memory;
 * `stream` is a cudaStream_t passed as void*; every function returns 0 on success and a non-zero status
 * otherwise, with a message retrievable through hvae_last_error().  Nothing here allocates or synchronises.
 *
 * Data layout in HBM:
 *   interactions  CSR over all users: indptr int64 [U+1], indices int32 [nnz] (sorted per row),
 *                 values float32 [nnz] or NULL (= all ones).  A batch is `rows` int32 [B] (user ids) or
 *                 NULL (= users 0..B-1).
 *   W1^T          encoder.0.weight held transposed, [N, ld1] float32, ld1 = round_up(h1, 4): one item's
 *                 row is contiguous (16-byte vector loads).
 *   activations   [B, ld] float32 with ld = round_up(width, 4), pad columns zero.
 *   E             item embeddings [N, d] float32 (exact mode) and/or bfloat16 (tensor-core mode).
 */
#ifndef HVAE_B200_H
#define HVAE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* Per-step scalars kept on the device so a captured CUDA graph replays unchanged. */
typedef struct hvae_step_state {
    int32_t adam_step;   /* number of optimiser steps taken (torch Adam's `step`) */
    int32_t anneal_step; /* AnnealedVAE.current_step, src/ml/model.py:310 */
    float step_size;     /* lr / (1 - beta1^step) */
    float bc2_sqrt;      /* sqrt(1 - beta2^step) */
    float beta_kl;       /* KL weight of this step */
    float inv_bg;        /* 1 / global batch size */
    float kl_coef;       /* beta_kl / global batch size */
    float clip_coef;     /* min(1, max_norm / (||g|| + 1e-6)) */
    float grad_norm;     /* ||g||_2 before clipping */
    float norm2;         /* ||g||_2^2 */
    uint32_t noise_lo;   /* 64-bit Philox counter base of the in-kernel dropout / eps noise, advanced per step */
    uint32_t noise_hi;
} hvae_step_state;

const char* hvae_last_error(void);
int hvae_abi_version(void);

/* ---- encoder (src/ml/model.py:111-127,149-153) ------------------------------------------------------ */
/* nn.Linear(N,h) on the sparse row as a gather-sum of W1^T rows + LayerNorm + GELU + Dropout.
 * gamma == NULL: plain linear output in `act`.  mask: uint8 keep-mask [B,h] or NULL (no dropout). */
int hvae_gather_ln_fwd(const int64_t* indptr, const int32_t* indices, const float* values, const int32_t* rows, int B,
                       const float* W1T, int ld, int h, const float* bias, const float* gamma, const float* beta,
                       const uint8_t* mask, float keep_scale, float* pre, float* mean, float* rstd, float* act,
                       void* stream);
/* LayerNorm + GELU + Dropout of a deeper hidden layer (model.py:115-117). */
int hvae_ln_act_fwd(const float* pre, int B, int h, int ld, const float* gamma, const float* beta, const uint8_t* mask,
                    float keep_scale, float* mean, float* rstd, float* act, void* stream);
/* autograd of the block above: d(pre), d(gamma), d(beta). */
size_t hvae_ln_bwd_workspace_floats(int B, int ld);
int hvae_ln_act_bwd(const float* dact, const float* pre, const float* mean, const float* rstd, const float* gamma,
                    const float* beta, const uint8_t* mask, float keep_scale, int B, int h, int ld, float* dpre,
                    float* dgamma, float* dbeta, float* workspace, void* stream);
/* column sums (bias gradients); workspace >= 64*C floats. */
int hvae_colsum(const float* X, int ld, int R, int C, float* out, float* workspace, void* stream);
/* d(W1^T) for the touched rows only (replaces the dense dW1 = dH^T X of autograd, SURVEY.md K1). */
/* Work plan: the touched items' entry lists are cut into work items of <= 64 entries (item popularity is heavy-tailed).
 * chunk_base, part_base: int32 [max_slots+1]; work_slot: int32 [hvae_w1_max_work(max_slots)]; multi_slot: int32
 * [hvae_w1_max_partial_rows(max_slots)] (slots with several chunks); n_work: int32 [2] = {work items, multi-chunk slots}. */
size_t hvae_w1_max_work(int max_slots);
size_t hvae_w1_max_partial_rows(int max_slots);
int hvae_w1_plan(const int32_t* seg_start, const int32_t* n_unique, int max_slots, int32_t* chunk_base, int32_t* part_base,
                 int32_t* work_slot, int32_t* multi_slot, int32_t* n_work, void* stream);
/* dpre: d(pre-activation) rows of the batch, [rows, ld]; or, for data-parallel training, the all-gathered per-rank
 * buffers read in place: row u lives at dpre + (u / block_rows) * block_stride + (u % block_rows) * ld
 * (block_rows <= 0: one plain matrix).  partial: [hvae_w1_max_partial_rows(max_slots), ld] scratch. */
int hvae_w1_grad(const int32_t* seg_start, const int32_t* n_unique, const int32_t* sorted_eid, const int32_t* ent_user,
                 const float* ent_val, int max_slots, const int32_t* chunk_base, const int32_t* part_base, const int32_t* work_slot,
                 const int32_t* multi_slot, const int32_t* n_work, const float* dpre, int ld, int block_rows, int64_t block_stride,
                 float* gs, float* partial, float* rownorm2, void* stream);
/* dense variant for the autograd-compatible path (atomics into a zeroed [N, ld] buffer). */
int hvae_w1_grad_dense(const int64_t* indptr, const int32_t* indices, const float* values, const int32_t* rows, int B,
                       const float* dpre, int ld, int h, float* dW1T, void* stream);

/* ---- batch plumbing ---------------------------------------------------------------------------------- */
size_t hvae_batch_temp_bytes(int cap, int n_items);
int hvae_batch_offsets(const int64_t* indptr, const int32_t* rows, int B, int32_t* boff, void* stream);
int hvae_batch_transpose(const int64_t* indptr, const int32_t* indices, const float* values, const int32_t* rows, int B,
                         int n_items, int cap, const int32_t* boff, int32_t* keys, int32_t* keys_sorted, int32_t* eid,
                         int32_t* eid_sorted, int32_t* head, int32_t* slot, int32_t* ent_user, float* ent_val,
                         int32_t* seg_start, int32_t* uniq_item, int32_t* slot_of_item, int32_t* n_unique,
                         int32_t* overflow, void* temp, size_t temp_bytes, void* stream);
/* Restores slot_of_item to -1 for the step's touched items.  `overflow` (may be NULL) is hvae_batch_transpose's counter of rows
 * that did not fit in `cap`: when non-zero the step's loss scalars `loss_out[0..2]` and accumulators `acc[0..2]` (may be NULL)
 * are set to NaN so that a too-small nnz bound can never pass silently; the counter itself is left for the host to read/clear. */
int hvae_batch_release(const int32_t* uniq_item, const int32_t* n_unique, int cap, int32_t* slot_of_item,
                       const int32_t* overflow, float* loss_out, float* acc, void* stream);

/* Host <-> device plumbing of the per-step API (one batch per call, as the reference's loop, train.py:86-96): the batch's CSR
 * slice from (pinned) host memory into the step's static device buffers (three async copies on `stream`), and n floats back
 * (async copy, then the call waits for `stream`). */
int hvae_h2d_csr_batch(const int64_t* h_crow, const int32_t* h_col, const float* h_val, int B, int64_t nnz, int64_t* d_crow,
                       int32_t* d_col, float* d_val, void* stream);
int hvae_d2h_floats(const float* d_src, int n, float* h_dst, void* stream);

/* ---- dense fp32 GEMM with arbitrary strides (aten::addmm / aten::mm, SURVEY.md K2,K5,K6,K8) ------------ */
int hvae_gemm_f32(int M, int N, int K, const float* A, int64_t a_rs, int64_t a_cs, const float* B, int64_t b_rs,
                  int64_t b_cs, float* C, int64_t ldc, const float* bias, float alpha, void* stream);

/* Same contract on the tensor cores (tcgen05 kind::tf32: fp32 operands read as TF32, fp32 accumulation in TMEM); used
 * for the MLP-stack GEMMs in bf16 mode.  Needs unit stride on one axis of A and of B, the other stride % 4 == 0 and
 * 16-byte aligned bases: hvae_gemm_tf32_supported() returns 1 when that holds. */
size_t hvae_gemm_tf32_supported(const float* A, int64_t a_rs, int64_t a_cs, const float* B, int64_t b_rs, int64_t b_cs);
int hvae_gemm_tf32(int M, int N, int K, const float* A, int64_t a_rs, int64_t a_cs, const float* B, int64_t b_rs,
                   int64_t b_cs, float* C, int64_t ldc, const float* bias, float alpha, void* stream);

/* The same tensor-core GEMM with the element-wise kernel that follows it in the model folded into its epilogue (one launch and one
 * round trip through HBM less each), and the bias gradient (column sums of what the epilogue wrote) added up in a fixed order by
 * the last m tile to finish.  `workspace`: hvae_gemm_colsum_workspace_floats(M, cols) floats, ZERO before the first use (the kernel
 * leaves its counters zero); `colsum` may be NULL.
 *   gelu_drop : pre = A B + bias ; act = gelu(pre) * mask * keep_scale          (model.py:90-93 projection_layer.0-2; ldc for both,
 *               columns N..ldc-1 are written as zeros)
 *   bf16      : C = A B + bias (C may be NULL) and its bf16 copy [M, ld_bf16] with zero padding (the user vectors that feed the
 *               scoring kernels, model.py:94,198)
 *   gelu_bwd  : dpre = (A B) * mask * keep_scale * gelu'(pre) ; colsum[n] = sum_m dpre[m, n]       (autograd of model.py:90-93)
 *   latent_bwd: dz = A B [M, L] -> dml = [dz + coef*mu | dz*eps*0.5*exp(0.5 logvar) + coef*0.5*(exp(logvar)-1)], colsum [2L]
 *               (autograd of model.py:157-179 + the KL term of model.py:286-287; same arithmetic as hvae_latent_bwd) */
size_t hvae_gemm_colsum_workspace_floats(int M, int cols);
int hvae_gemm_tf32_gelu_drop(int M, int N, int K, const float* A, int64_t a_rs, int64_t a_cs, const float* B, int64_t b_rs,
                             int64_t b_cs, float* pre, float* act, int64_t ldc, const float* bias, const uint8_t* mask,
                             float keep_scale, void* stream);
int hvae_gemm_tf32_bf16(int M, int N, int K, const float* A, int64_t a_rs, int64_t a_cs, const float* B, int64_t b_rs,
                        int64_t b_cs, float* C, int64_t ldc, const float* bias, void* C_bf16, int64_t ld_bf16, void* stream);
int hvae_gemm_tf32_gelu_bwd(int M, int N, int K, const float* A, int64_t a_rs, int64_t a_cs, const float* B, int64_t b_rs,
                            int64_t b_cs, float* dpre, int64_t ldc, const float* pre, const uint8_t* mask, float keep_scale,
                            float* colsum, float* workspace, void* stream);
int hvae_gemm_tf32_latent_bwd(int M, int L, int K, const float* A, int64_t a_rs, int64_t a_cs, const float* B, int64_t b_rs,
                              int64_t b_cs, const float* ml, int64_t ldml, const float* eps, const float* coef, float* dml,
                              float* colsum, float* workspace, void* stream);

/* ---- latent (model.py:157-179, 92-93, 281-290) -------------------------------------------------------- */
int hvae_reparam_kl(const float* ml, int ldml, const float* eps, int B, int L, float* z, int ldz, float* kl_row,
                    void* stream);
int hvae_latent_bwd(const float* dz, int lddz, const float* ml, int ldml, const float* eps, int B, int L,
                    const float* coef, float* dml, void* stream);
int hvae_gelu_drop_fwd(const float* q, const uint8_t* mask, float keep_scale, int B, int d, int ld, float* t, void* stream);
int hvae_gelu_drop_bwd(const float* dt, const float* q, const uint8_t* mask, float keep_scale, int B, int d, int ld,
                       float* dq, void* stream);
int hvae_loss_finalize(const float* lse, const float* dot, const float* xsum, const float* kl_row, int B,
                       const float* inv_bg, const float* beta, float* out, float* acc, void* stream);

/* ---- scoring rows (model.py:198,281; evaluate.py:143-146) ---------------------------------------------- */
int hvae_row_lse(const float* S, int64_t lds, int rows, int N, float* lse, void* stream);
int hvae_row_softmax_scale(float* S, int64_t lds, int rows, int N, const float* lse, const float* xsum,
                           const float* inv_bg, void* stream);
int hvae_sparse_dot_xsum(const int64_t* indptr, const int32_t* indices, const float* values, const int32_t* rows, int B,
                         const void* U, int ldu, const void* E, int lde, int d, int is_bf16, float* dot, float* xsum,
                         void* stream);
/* dU = s_b * O_b - (1/Bg) * sum_j x_bj E_idx_j;  O: n_parts partial sums [n_parts][B][ldo];
 * s_b = oscale ? oscale[b]/Bg : 1 (oscale = row sums |x|_b when O holds softmax-weighted sums).
 * O_b = sum_p O[p][b], or sum_p w_part[p][b] O[p][b] for the unnormalised partials of hvae_tc_score_onepass
 * (w_part [n_parts][B] from hvae_tc_onepass_combine; NULL otherwise). */
int hvae_du_finalize(const int64_t* indptr, const int32_t* indices, const float* values, const int32_t* rows, int B,
                     const float* O, int ldo, int n_parts, const float* oscale, const float* w_part, const void* E, int lde,
                     int d, int is_bf16, const float* inv_bg, float* dU, int lddu, void* stream);
/* The same directly after hvae_tc_score_onepass, with hvae_tc_onepass_combine folded in (one launch less on the step's critical
 * path): c_part [n_parts, B], l_part [n_parts, n_sub, B] are the kernel's per-split shifts and numerator sums; writes lse [B]. */
int hvae_du_finalize_onepass(const int64_t* indptr, const int32_t* indices, const float* values, const int32_t* rows, int B,
                             const float* O, int ldo, int n_parts, const float* oscale, const float* c_part,
                             const float* l_part, int n_sub, float* lse, const void* E, int lde, int d, int is_bf16,
                             const float* inv_bg, float* dU, int lddu, void* stream);
/* Seen-item masking (in place) + top-K of materialised scores under the order (score desc, index desc).  Rows are cut into
 * hvae_mask_topk_chunks(n_rows, N) column chunks; cand_val / cand_idx: scratch [n_rows, chunks * K] (NULL if chunks == 1). */
size_t hvae_mask_topk_chunks(int n_rows, int N);
int hvae_mask_topk(float* S, int64_t lds, int n_rows, int N, int item_offset, const int64_t* indptr,
                   const int32_t* indices, const int32_t* rows, int exclude_seen, int K, float* cand_val, int32_t* cand_idx,
                   float* out_val, int32_t* out_idx, void* stream);
/* The same with per-row item allow-sets: allow is [F, allow_stride_words] bitmaps over global item ids (bit i set = item i may
 * be returned, allow_stride_words >= ceil((item_offset + N) / 32)), allow_of_row [n_rows] picks a row's bitmap (-1 =
 * unrestricted).  allow == NULL is hvae_mask_topk.  Slots a row cannot fill hold (-inf, -1). */
int hvae_mask_topk_filtered(float* S, int64_t lds, int n_rows, int N, int item_offset, const int64_t* indptr,
                            const int32_t* indices, const int32_t* rows, int exclude_seen, const uint32_t* allow,
                            int64_t allow_stride_words, const int32_t* allow_of_row, int K, float* cand_val, int32_t* cand_idx,
                            float* out_val, int32_t* out_idx, void* stream);
int hvae_topk_merge(const float* cval, const int32_t* cidx, int n_rows, int GK, int K, float* out_val, int32_t* out_idx,
                    void* stream);
/* The same merge over the blocks of an all-gather, read in place: rank g's K candidates of row r are at
 * cval/cidx[g * group_stride + r * K] (item-sharded evaluation: local top-K -> all-gather -> merge, SURVEY.md §8e). */
int hvae_topk_merge_groups(const float* cval, const int32_t* cidx, int n_rows, int n_groups, int64_t group_stride, int K,
                           float* out_val, int32_t* out_idx, void* stream);
/* Negative-sampling protocol (evaluate.py:149-185): scores of C candidates per row (candidate 0 = test item) and the
 * 0-based rank of candidate 0 under a stable descending sort.  cand: int32 [B, C]; scores may be NULL. */
int hvae_candidate_rank(const void* U, int ldu, const void* E, int lde, int d, int is_bf16, const int32_t* cand, int C, int B,
                        float* scores, int32_t* rank, void* stream);
/* Recall/NDCG/HR@K (evaluate.py:32-54,90-98) */
int hvae_hit_mask(const int32_t* topk, int n_rows, int K, const int64_t* rel_ptr, const int32_t* rel_idx, uint32_t* mask,
                  void* stream);
int hvae_metrics_reduce(const uint32_t* mask, const int64_t* rel_ptr, int n_rows, const int32_t* kvals, int nk,
                        const double* disc, const double* idcg, double* workspace, double* out, void* stream);

/* ---- tensor-core scoring, bf16 mode (model.py:198,281; evaluate.py:125-147) ------------------------------ */
/* S = U E^T on tcgen05 (TMA-fed, TMEM accumulators); the [B,N] scores never reach HBM.  U: bf16 [B, ldu],
 * E: bf16 [N, lde]; ldu, lde multiples of 8, columns d..ld zero. */
int hvae_cast_bf16(const float* src, int rows, int cols, int ld_src, void* dst_bf16, int ld_dst, void* stream);
size_t hvae_tc_n_splits(int B, int N);
/* lse[b] = log sum_i exp(S_bi).  workspace >= 2 * B * hvae_tc_n_splits(B,N) floats. */
int hvae_tc_score_lse(const void* U, int ldu, int B, const void* E, int lde, int N, int d, float* lse, float* workspace,
                      void* stream);
size_t hvae_tc_topk_splits(int B, int N);
/* per item split, the K best (score, global item id) of every user with the user's seen items excluded
 * (indptr == NULL: nothing excluded).  cand_val / cand_idx: [B, hvae_tc_topk_splits(B,N) * K]; reduce with
 * hvae_topk_merge.  K <= 32.  E points at the first item of the shard, item_offset is its global id. */
int hvae_tc_score_topk(const void* U, int ldu, int B, const void* E, int lde, int N, int d, int item_offset,
                       const int64_t* indptr, const int32_t* indices, const int32_t* rows, int K, float* cand_val,
                       int32_t* cand_idx, void* stream);
/* The same with per-row item allow-sets (bitmaps as in hvae_mask_topk_filtered, over global ids: a shard's item_offset need
 * not be a multiple of 32).  allow == NULL is hvae_tc_score_topk.  Slots a row cannot fill hold (-inf, -1). */
int hvae_tc_score_topk_filtered(const void* U, int ldu, int B, const void* E, int lde, int N, int d, int item_offset,
                                const int64_t* indptr, const int32_t* indices, const int32_t* rows,
                                const uint32_t* allow, int64_t allow_stride_words, const int32_t* allow_of_row,
                                int K, float* cand_val, int32_t* cand_idx, void* stream);

/* Backward through the scores: O[b,:] = sum_i softmax(S_b)_i E_i with S recomputed on the tensor cores
 * (autograd of model.py:198,281; E is a frozen buffer, no dE).  lse from hvae_tc_score_lse.
 * Opart: [hvae_tc_grad_splits(B,N,d)][B][ldo] partial sums over item splits. */
size_t hvae_tc_grad_splits(int B, int N, int d);
/* Diagnostic: CTA pairs (clusters of 2) of the cta_group::2 scoring kernel the device holds at once with smem_bytes of dynamic
 * shared memory per CTA (0 = the kernel's own size); < 0 = query failed. */
int hvae_tc_duo_max_clusters(int smem_bytes);
/* Profiling: while trace != NULL the cta_group::2 scoring kernel runs an instrumented build that writes per CTA and role
 * (TMA producer, MMA issuer, softmax warp) 8 int64 cycle counters of its barrier waits: [2 * m_tiles * n_splits][3][8]. */
int hvae_tc_duo_trace(int64_t* trace);
int hvae_tc_score_grad(const void* U, int ldu, int B, const void* E, int lde, int N, int d, const float* lse, float* Opart,
                       int ldo, void* stream);

/* hvae_tc_score_lse + hvae_tc_score_grad as two launches (the backward kernel merges the forward's partial
 * max / sum-exp itself and publishes lse). */
int hvae_tc_score_lse_grad(const void* U, int ldu, int B, const void* E, int lde, int N, int d, float* lse, float* workspace,
                           float* Opart, int ldo, void* stream);

/* Forward + backward through the scores in ONE sweep over the items (what a training step uses; 4BNd executed flops instead
 * of 6BNd): softmax numerators are taken against a per-row shift that does not depend on the scores (0 to begin with), so no
 * forward pass has to come first; a row whose numerator sum leaves the range in which fp32/bf16 lose nothing (scores beyond
 * about +-70) makes its CTA repeat the sweep with the shift moved by 60.
 * Out: Opart [S = hvae_tc_grad_splits(B,N,d)][B][ldo] UNNORMALISED partial sums; c_part [S][B] the shift each split ended up
 * with; l_part [S][n_sub = hvae_tc_onepass_subparts(d)][B] row sums of the numerators.
 * hvae_tc_onepass_combine: lse_b = log sum_p e^{c_p} l_p and the weights w_part [S][B] = e^{c_p} / sum_q e^{c_q} l_q that
 * hvae_du_finalize applies (O_b = sum_p w_part[p][b] Opart[p][b]). */
size_t hvae_tc_onepass_subparts(int d);
int hvae_tc_score_onepass(const void* U, int ldu, int B, const void* E, int lde, int N, int d, float* c_part, float* l_part,
                          float* Opart, int ldo, void* stream);
int hvae_tc_onepass_combine(const float* c_part, const float* l_part, int n_parts, int n_sub, int B, float* lse,
                            float* w_part, void* stream);

/* ---- optimiser (train.py:63,88-92; model.py:312-323) --------------------------------------------------- */
/* advance != 0: a training step (Adam step count, annealing step and the noise counter (+= noise_stride) move on) */
int hvae_step_begin(hvae_step_state* state, double lr, double beta1, double beta2, double kl_beta_min, double kl_beta_max,
                    int anneal_steps, int b_global, int advance, uint32_t noise_stride, void* stream);
int hvae_grad_norm_clip(const float* gdense, int64_t n_dense, const float* rownorm2, const int32_t* n_unique,
                        float max_norm, hvae_step_state* state, float* workspace, void* stream);
/* The same in two calls (identical arithmetic): the sum of squares of the dense gradients depends on them only and can run beside
 * the layer-1 weight-gradient kernels; the finish adds the rows' squared norms and writes the clip coefficient. */
int hvae_grad_sumsq_dense(const float* gdense, int64_t n_dense, float* workspace, void* stream);
int hvae_grad_norm_finish(int64_t n_dense, const float* rownorm2, const int32_t* n_unique, float max_norm,
                          hvae_step_state* state, const float* workspace, void* stream);
int hvae_adam_step(float* params, float* exp_avg, float* exp_avg_sq, int64_t n_params, int64_t n_w1, int ld1,
                   const int32_t* slot_of_item, const float* gsparse, const float* gdense, const hvae_step_state* state,
                   float weight_decay, float beta1, float beta2, float eps, void* stream);
/* The same update in two calls, bit for bit: (1) the W1^T rows WITHOUT a gradient in this step -- their update needs only slot_of_item of
 * the step's batch and the step scalars, so a step runs it beside its backward pass (2.9 GB of the optimiser's traffic off the critical
 * path); (2) the rows with a gradient (compact row k of gsparse = item uniq_item[k], k < *n_unique <= max_rows) and the dense tensors. */
int hvae_adam_step_untouched(float* params, float* exp_avg, float* exp_avg_sq, int64_t n_w1, int ld1,
                             const int32_t* slot_of_item, const hvae_step_state* state, float weight_decay, float beta1,
                             float beta2, float eps, void* stream);
int hvae_adam_step_touched(float* params, float* exp_avg, float* exp_avg_sq, int64_t n_params, int64_t n_w1, int ld1,
                           const int32_t* uniq_item, const int32_t* n_unique, int max_rows, const float* gsparse,
                           const float* gdense, const hvae_step_state* state, float weight_decay, float beta1, float beta2,
                           float eps, void* stream);
/* Counter-based (Philox4x32-10) keep-masks / standard normals; counter = offset + state->noise (state may be NULL). */
int hvae_fill_noise(uint8_t* mask, int64_t n_mask, float keep_prob, float* eps, int64_t n_eps, uint64_t seed,
                    uint64_t offset, uint32_t stream_id, const hvae_step_state* state, void* stream);

/* ---- data-parallel gradient exchange over NVLink / NVSwitch (new; the reference is single-process) ------------------- */
/* One-shot all-gather by direct stores into every rank's symmetric receive buffer (NVSwitch multicast when mc_dst != NULL,
 * else the `world` unicast peer mappings in peer_ptrs).  The caller brackets it with symmetric-memory barriers. */
int hvae_nvl_push(const float* src, int64_t n, float* mc_dst, const uint64_t* peer_ptrs, int world, int64_t dst_off,
                  void* stream);

/* ---- Mult-VAE baseline (src/ml/baseline.py:126-231) -- the kernels only that model needs; the rest of it runs on the entry
 * points above (gather-sum, GEMMs, reparameterise/KL, materialised scoring, item-major gradient reduction, Adam) ------------- */
/* Input transform on the sparse row: F.normalize(x, p=2, dim=1) then input dropout (baseline.py:151) as per-entry values
 * out[j] = x_j / max(||x_b||, 1e-12) * keep_j * keep_scale, written at the entries' positions in the global CSR (out has the
 * CSR's nnz floats).  keep (may be NULL): uint8 flags in batch order, keep_ptr[b] = offset of batch row b's first entry. */
int hvae_mv_input_values(const int64_t* indptr, const float* values, const int32_t* rows, int B, const uint8_t* keep,
                         const int32_t* keep_ptr, float keep_scale, float* out, void* stream);
/* t[B, ldt] = dropout(tanh(q[B, ldq])) over d columns (mask may be NULL), pad columns 0; ones_col >= d: t[:, ones_col] = 1. */
int hvae_tanh_drop_fwd(const float* q, const uint8_t* mask, float keep_scale, int B, int d, int ldq, float* t, int ldt,
                       int ones_col, void* stream);
/* dq[B, ldq] = dt[B, lddt] * mask * keep_scale * (1 - tanh(q)^2) */
int hvae_tanh_drop_bwd(const float* dt, int lddt, const float* q, const uint8_t* mask, float keep_scale, int B, int d, int ldq,
                       float* dq, void* stream);
/* dst[item[s], 0:cols] += alpha * src[s, 0:cols] for s < *n_rows (<= max_rows). */
int hvae_rows_axpy(const int32_t* item, const int32_t* n_rows, int max_rows, const float* src, int ld_src, float alpha,
                   float* dst, int ld_dst, int cols, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* HVAE_B200_H */
