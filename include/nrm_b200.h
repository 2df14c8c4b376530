/*
 * nrm_b200.h -- C ABI of libnrm_b200.so: the B200 (sm_100a) hot path of the EB-NeRD
 * news recommender (ChuhanZhou/News_Recommendation_Model).
 *
 * The reference has no FFI: its hot path is Python calling torch.nn modules.  The
 * entry points below are what a binding for that path binds, one per reference call
 * site; every one takes plain device pointers and sizes, allocates nothing, never
 * synchronises, and enqueues all of its work on `stream` (a training forward also forks a
 * library-owned side stream from `stream` for the id sort the backward needs; nrm_backward
 * joins it back, so callers only ever see `stream` -- CUDA-graph capture included).
 *
 *   reference call (file:line)                               entry point
 *   ------------------------------------------------------   -------------------------
 *   UserModel.forward         models/user_model.py:27-35      nrm_forward
 *     UserInvariantInterestModel.forward
 *                 models/user_invariant_interest_model.py:73-88   (inside nrm_forward)
 *     PointwiseAttentionExpanded.forward
 *                 models/attention_model.py:52-97             (inside nrm_forward)
 *     UserInstantInterestModel.forward
 *                 models/user_instant_interest_model.py:20-23 (inside nrm_forward)
 *   s_label / s_ti            user_invariant_interest_model.py:83-87   nrm_forward_scores, nrm_history_topk
 *   ensemble softmax + order  test.py:58-63, 124-127 over a shared pool  nrm_forward_pool, nrm_pool_topk
 *   UserModel.loss            models/user_model.py:37-43      nrm_loss_forward
 *   loss.backward()           train.py:73                     nrm_loss_backward, nrm_backward
 *   optimizer.step()          train.py:48,74                  nrm_adam_step
 *
 * Conventions
 *   - all pointers are DEVICE pointers unless named host_*; `stream` is a cudaStream_t
 *     passed as void* (0 = legacy default stream);
 *   - every function returns 0 on success or a negative NRM_E* code; nrm_last_error()
 *     returns a thread-local description of the last failure;
 *   - feature tensors are the reference's packed float64 rows
 *       x_history [B,H,80], x_target [B,C,78], x_global [B,C,3]
 *     (models/user_invariant_interest_model.py:14-22); x_target / x_global may be
 *     column-trimmed views as produced by test.py:53-54, hence the batch strides
 *     (in elements); rows inside one impression are contiguous;
 *   - parameters live in ONE flat float32 buffer whose layout is given by the
 *     nrm_layout_* functions (state_dict order of the reference, 16-byte aligned
 *     entries, `delta` last); gradients use the same layout;
 *   - `precision` selects how the pairwise attention products (forward and backward) are
 *     evaluated; everything else is fp32 in every mode:
 *       0 = fp32    FFMA on the CUDA cores (bit-for-bit fp32 products);
 *       1 = bf16    tcgen05 tensor-core tiles, operands rounded to bf16, fp32 accumulation;
 *       2 = bf16x3  tcgen05 tiles with every operand split in hi + lo bf16 parts and three
 *                   products per tile (a_hi b_hi + a_hi b_lo + a_lo b_hi), fp32 accumulation:
 *                   relative operand error 2^-16 (torch's float32 matmul precision "high");
 *                   meets the fp32 parity tolerances of tests/parity.py.
 */
#ifndef NRM_B200_H
#define NRM_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NRM_OK            0
#define NRM_EINVAL       -1   /* bad argument (null pointer, non-positive size, ...) */
#define NRM_EWORKSPACE   -2   /* workspace too small or misaligned                    */
#define NRM_ECUDA        -3   /* a CUDA runtime call or kernel launch failed          */
#define NRM_EUNSUPPORTED -4   /* configuration not built into this library           */

#define NRM_PRECISION_FP32 0
#define NRM_PRECISION_BF16 1
#define NRM_PRECISION_BF16X3 2

/* `mode` bit flags of the forward/backward entry points */
#define NRM_MODE_BN_BATCH_STATS 1   /* module.training: BatchNorm uses (and records) batch statistics */
#define NRM_MODE_KEEP_FOR_BWD   2   /* keep activations / sort keys in the workspace for nrm_backward  */
#define NRM_MODE_EVAL           0
#define NRM_MODE_TRAIN          3

int         nrm_version(void);
const char* nrm_last_error(void);

/* ---- instrumentation (bench.py) --------------------------------------------------- */
/* Kernels launched by this library in this process so far. */
unsigned long long nrm_launch_count(void);
/* While enabled, the major kernel groups are bracketed with CUDA events on their launch
 * stream; nrm_timing_report writes one "name count total_ms" line per group into buf
 * (synchronising on the recorded events) and returns 0.  Enabling resets the counters. */
void        nrm_timing_enable(int on);
int         nrm_timing_report(char* buf, size_t buf_bytes);
/* Self test of the tcgen05 building blocks used by the tensor-core paths: out[q] (q = 0,1;
 * [64,64] fp32) from a_q / b_q [64,64] fp32 row-major with fp32 accumulation.
 * mode 0: a_q b_q^T (both operands K-major); 1: a_q^T b_q (both read MN-major);
 * 2: a_q b_q (A K-major, B MN-major).  split 1: operands rounded to bf16; 3: hi/lo split.
 * Exercises descriptor encoding for both majors, TMEM allocation, the half-lane accumulator
 * pairing, mbarrier completion and tcgen05.ld. */
int         nrm_debug_umma_selftest(const float* a0, const float* a1, const float* b0, const float* b1,
                                    float* out, int mode, int split, void* stream);

/* Cycle counts of back-to-back tcgen05 products (tools/mma_microbench.py): out[0] = issue cycles, out[1] = cycles
 * until the mbarrier completes.  variant 0: M64 N64 K-major; 1: M64 N64 MN-major; 2: M128 N64; 3: M64 N8;
 * 4: tcgen05.ld only.  `reps` products of `nk` K=16 steps each. */
int         nrm_debug_mma_microbench(long long* out, int variant, int reps, int nk, void* stream);

/* ---- data parallelism over peer memory (no counterpart in the single-process reference; north_star: gradient all-reduce) ----
 * The gradient average over the ranks is fused into the optimizer: every rank's flat gradient buffer sits in symmetric (peer-mapped)
 * memory and nrm_adam_step_allreduce reads all of them in rank order while it updates.  `peer_ctx` is a device struct
 *     { int rank, world; long long n; const float* grad[8]; unsigned* pad[8]; double* stats[8];
 *       const long long* suid[8]; const float* sval[8]; long long* acc; unsigned* gridbar; long long delta_off, delta_n, rows; }
 * (nrm_peer_ctx_bytes() bytes) holding the peer-mapped pointers; the library uses the u32 words [64, nrm_peer_flag_words()) of every
 * signal pad; `stats` buffers hold nrm_peer_stats_bytes() bytes.  Call order per step: ... forward, loss ..., nrm_peer_wait_consumed,
 * backward ..., nrm_adam_step_allreduce.  nrm_peer_allsum_stats sums the BatchNorm statistics (which = 0 forward, 1 backward) over the
 * ranks between the two halves of nrm_forward / nrm_backward (synchronised BatchNorm). */
size_t      nrm_peer_ctx_bytes(void);
size_t      nrm_peer_stats_bytes(void);
int         nrm_peer_flag_words(void);
int         nrm_peer_preload(void);
int         nrm_adam_step_allreduce(float* param, float* exp_avg, float* exp_avg_sq, long long n, void* adam_state,
                                    const void* peer_ctx, void* ticket, void* stream);
/* Large user tables (user_num ~ 2 000 000): the per-user bias gradient travels as (user id, value) per impression instead of a dense
 * [user_num + 1] buffer: nrm_loss_backward_sparse publishes the lists (symmetric memory), nrm_adam_step_allreduce sums all ranks' lists into
 * peer_ctx->acc (fixed point, integer atomics: order independent) and runs the dense Adam pass over delta from it (delta_n > 0). */
int         nrm_loss_backward_sparse(const long long* user_id, int B, int C, const float* grad_loss, float* dlogits, long long delta_numel,
                                     long long* sparse_uid, float* sparse_val, const void* scratch, size_t scratch_bytes, void* stream);
int         nrm_peer_wait_consumed(const void* adam_state, const void* peer_ctx, void* stream);
int         nrm_peer_allsum_stats(const double* local, int which, double* out, const void* adam_state, const void* peer_ctx, void* stream);

int         nrm_debug_rsprof(long long* host_out64);   /* row-stacked attention kernels: per-role wait cycles (-DNRM_RS_PROFILE builds) */
long long   nrm_debug_ws_field(int B, int H, int C, int mode, const char* name, long long* bytes);   /* byte offset of a workspace buffer (debugging) */
int         nrm_debug_headprof(long long* host_out32); /* tensor-core head kernels: the same (-DNRM_RS_PROFILE builds) */

/* ---- flat parameter layout (reference state_dict order; SURVEY.md section 8b) ---- */
int         nrm_layout_entries(void);                 /* trainable tensors incl. delta     */
const char* nrm_layout_name(int i);                   /* reference state_dict key          */
long long   nrm_layout_offset(int i);                 /* offset in floats                  */
long long   nrm_layout_numel(int i);                  /* element count (-1: delta, runtime)*/
long long   nrm_layout_fixed_floats(void);            /* floats before delta (16B padded)  */

/* ---- workspace ------------------------------------------------------------------- */
/* Bytes of scratch nrm_forward/nrm_backward need for one (B,H,C) batch.  With
 * NRM_MODE_KEEP_FOR_BWD in `mode` it is sized for forward + backward (activations are kept
 * between the two calls). */
size_t nrm_workspace_bytes(int B, int H, int C, int mode);
/* byte offset of e_concat [B*C,264] (= [eu_H 128 | eu_L 8 | ec 128], user_model.py:31) inside that workspace: the output of
 * nrm_forward_encoder (UserInvariantInterestModel.forward + UserInstantInterestModel.forward) */
size_t nrm_workspace_e_offset(int B, int H, int C, int mode);

/* ---- UserModel.forward (user_model.py:27-35) ------------------------------------- */
/* mode & NRM_MODE_BN_BATCH_STATS: BatchNorm uses batch statistics, updates
 * bn_running_mean/var (momentum 0.1, unbiased variance) and increments
 * *bn_num_batches_tracked; otherwise it uses the running statistics (module.eval()).
 * mode & NRM_MODE_KEEP_FOR_BWD: keeps what nrm_backward needs in `workspace`.
 * logits: [B,C] float32. */
int nrm_forward(const double* x_history, const double* x_target, long long x_target_batch_stride,
                const double* x_global, long long x_global_batch_stride,
                int B, int H, int C,
                const float* params, float* bn_running_mean, float* bn_running_var,
                long long* bn_num_batches_tracked,
                int mode, int precision,
                float* logits, void* workspace, size_t workspace_bytes, void* stream);

/* Two-phase variant for synchronised BatchNorm across data-parallel ranks:
 * nrm_forward_encoder writes e_concat and bn_sums[2][264] (double: column sums and sums
 * of squares over this rank's B*C rows, may be null to keep them in the workspace only);
 * the caller all-reduces bn_sums and calls nrm_forward_head with the GLOBAL row count
 * (bn_sums null / bn_global_rows 0 = use this rank's own statistics).  `precision` is the one given to
 * nrm_forward_encoder (it selects the tensor-core head, whose weight images that call prepares). */
int nrm_forward_encoder(const double* x_history, const double* x_target, long long x_target_batch_stride,
                        const double* x_global, long long x_global_batch_stride,
                        int B, int H, int C, const float* params, int mode, int precision,
                        double* bn_sums, void* workspace, size_t workspace_bytes, void* stream);
int nrm_forward_head(int B, int H, int C, const float* params, float* bn_running_mean, float* bn_running_var,
                     long long* bn_num_batches_tracked, int mode, int precision,
                     const double* bn_sums, long long bn_global_rows,
                     float* logits, void* workspace, size_t workspace_bytes, void* stream);

/* ---- backward of UserModel.forward (loss.backward(), train.py:73) ---------------- */
/* dlogits [B,C] float32.  Writes the gradient of every trainable tensor except `delta`
 * into `grads` (flat layout, overwritten, not accumulated).  Must follow an
 * nrm_forward(mode & NRM_MODE_KEEP_FOR_BWD) on the same inputs and workspace.
 * Two-phase variant for synchronised BatchNorm: nrm_backward_head stops after writing
 * bn_bwd_sums[2][264] (double: column sums of dL/dxhat and dL/dxhat*xhat); the caller
 * all-reduces them and calls nrm_backward_encoder. */
int nrm_backward(const double* x_history, const double* x_target, long long x_target_batch_stride,
                 const double* x_global, long long x_global_batch_stride,
                 int B, int H, int C, const float* params, int mode, int precision,
                 const float* dlogits, float* grads,
                 void* workspace, size_t workspace_bytes, void* stream);
int nrm_backward_head(int B, int H, int C, const float* params, int precision, const float* dlogits, float* grads,
                      double* bn_bwd_sums, void* workspace, size_t workspace_bytes, void* stream);
/* As nrm_backward_head, but the head's five weight gradients (needed by the optimizer only) are left running on the
 * library's side stream of `stream`; the NEXT nrm_backward_encoder on the same stream joins them before it returns, so
 * `grads` is complete after that call as usual.  For callers that put a cross-rank exchange of the BatchNorm sums
 * between the two calls (FusedTrainStep with synchronised BatchNorm); a caller that reads the head's weight gradients
 * between the calls (bucketed all-reduce, engine.backward_params) uses nrm_backward_head. */
int nrm_backward_head_deferred(int B, int H, int C, const float* params, int precision, const float* dlogits, float* grads,
                               double* bn_bwd_sums, void* workspace, size_t workspace_bytes, void* stream);
int nrm_backward_encoder(const double* x_history, const double* x_target, long long x_target_batch_stride,
                         const double* x_global, long long x_global_batch_stride,
                         int B, int H, int C, const float* params, int mode, int precision,
                         const double* bn_bwd_sums, long long bn_global_rows, float* grads,
                         void* workspace, size_t workspace_bytes, void* stream);

/* ---- the compact wire format as a direct input (no expansion to the packed float64 tensors) ----------------------------
 * nrm_expand_compact (below) rebuilds the reference's packed tensors for the entry points above.  These variants hand the
 * article table + per-impression ids / time buckets / click features straight to the row kernels instead: the 36 MB of
 * float64 rows are neither written nor read.  Same results, bit for bit.  Tensor-core precisions only (the FFMA attention
 * kernels of precision fp32 read the packed rows): NRM_EUNSUPPORTED otherwise.  label32 / label64 are optional (both null):
 * when given, the float32 labels are converted to the float64 labels nrm_loss_forward reads. */
typedef struct {
  const float* articles; int n_articles;      /* [n,80] float32, row 0 = the all-zero pad article                 */
  const int* hist_article; const unsigned* hist_time; const float* hist_click;   /* [B,H], [B,H] packed buckets, [B,H,2] */
  const int* cand_article; const unsigned* cand_time;                            /* [B,C], [B,C]                          */
  const float* label32; double* label64;      /* [B,C] each, optional                                              */
} nrm_compact_batch;
int nrm_forward_compact(const nrm_compact_batch* batch, int B, int H, int C, const float* params, float* bn_running_mean,
                        float* bn_running_var, long long* bn_num_batches_tracked, int mode, int precision,
                        float* logits, void* workspace, size_t workspace_bytes, void* stream);
int nrm_forward_encoder_compact(const nrm_compact_batch* batch, int B, int H, int C, const float* params, int mode, int precision,
                                double* bn_sums, void* workspace, size_t workspace_bytes, void* stream);
int nrm_backward_compact(const nrm_compact_batch* batch, int B, int H, int C, const float* params, int mode, int precision,
                         const float* dlogits, float* grads, void* workspace, size_t workspace_bytes, void* stream);
int nrm_backward_encoder_compact(const nrm_compact_batch* batch, int B, int H, int C, const float* params, int mode, int precision,
                                 const double* bn_bwd_sums, long long bn_global_rows, float* grads, void* workspace,
                                 size_t workspace_bytes, void* stream);

/* ---- attention scores: "which past clicks made the model rank this article high?" -------------------------------------------
 * The pairwise attention scores s[c][h] of both branches (PointwiseAttentionExpanded.forward, attention_model.py:52-97, called at
 * user_invariant_interest_model.py:83-87: label_attention, text_img_attention) for every (candidate, history row) pair, computed by
 * the kernels that compute the logits.  scores: float32 [2,B,C,H], branch 0 = label_attention, 1 = text_img_attention.  Pad history
 * rows get scores too (the reference does not mask them; they contribute to the pooled sum).
 *   nrm_forward_scores[_compact]: nrm_forward[_compact] in mode NRM_MODE_EVAL (any other mode: NRM_EINVAL; BatchNorm reads its
 *     running statistics and nothing is written to them) that also writes `scores`; the logits are bit-identical to nrm_forward's
 *     for the same precision, the workspace is nrm_workspace_bytes(B, H, C, NRM_MODE_EVAL).  The compact variant has
 *     nrm_forward_compact's precision limits.
 *   nrm_history_topk: per (branch, b, c) row the k largest scores and their history positions, descending, ties to the lower
 *     position (Python's stable sorted(..., reverse=True)); idx_out int32 / val_out float32 [2,B,C,k], 1 <= k <= min(H, 64).  Pad rows
 *     are left out: all-zero rows of x_history [B,H,80] or hist_article [B,H] == 0 (at most one of the two; both null: none); slots
 *     beyond the real rows get index -1 and score NaN. */
int nrm_forward_scores(const double* x_history, const double* x_target, long long x_target_batch_stride,
                       const double* x_global, long long x_global_batch_stride, int B, int H, int C,
                       const float* params, float* bn_running_mean, float* bn_running_var, long long* bn_num_batches_tracked,
                       int mode, int precision, float* logits, float* scores, void* workspace, size_t workspace_bytes, void* stream);
int nrm_forward_scores_compact(const nrm_compact_batch* batch, int B, int H, int C, const float* params, float* bn_running_mean,
                               float* bn_running_var, long long* bn_num_batches_tracked, int mode, int precision,
                               float* logits, float* scores, void* workspace, size_t workspace_bytes, void* stream);
int nrm_history_topk(const float* scores, int B, int C, int H, int k, const double* x_history, const int* hist_article,
                     int* idx_out, float* val_out, void* stream);

/* ---- recommendation: every user against a shared pool of N articles -------------------------------------------------------------
 * The other way round from the [B,C] impressions above: score all N articles of a pool (e.g. the articles live now) for each of B
 * users and keep each user's k best unread ones.
 *   nrm_forward_pool: logits [B,N] float32; logits[b][n] is, bit for bit, what nrm_forward in mode NRM_MODE_EVAL returns for
 *     impression b with the user's history and the whole pool as its candidates (x_target[b] / x_global[b] = the pool's rows for
 *     every b), in the same precision (all three).  BatchNorm reads its running statistics only.
 *     users->hist_* are the users' [B,H] / [B,H,2] compact histories; users->cand_article / cand_time are the pool's [N] ids and
 *     packed time buckets (one time for all users); label32 / label64 must be null.  The pool is processed in chunks of `chunk`
 *     articles (a positive multiple of 8, the attention's candidate group: any such chunk gives the same bits); the workspace
 *     is nrm_pool_workspace_bytes(B, H, N, chunk) bytes, 256-byte aligned, and grows with B * chunk.
 *   nrm_pool_topk: per user b the k pool positions with the largest score, descending, ties to the lower position (Python's
 *     stable sorted(..., reverse=True), test.py:124-127); pos_out int32 / val_out float32 [B,k], 1 <= k <= min(N, 1024).
 *     logits: n_models >= 1 (at most 16) stacked [B,N] slices, model m at logits + m * model_stride.  Position n is eligible
 *     unless pool_article[n] is 0 or outside [1, n_articles), a logit of n is NaN in any model, or (hist_article [B,H] given;
 *     null = no exclusion) pool_article[n] equals one of the user's non-pad history ids.  Score: the logit for one model; for
 *     n_models >= 2 the mean over the models of the softmax over the user's eligible positions (test.py:58-63),
 *     (1/M) sum_m exp(x_m - max_m) / sum_eligible exp(x_m - max_m), in float32.  Slots beyond the eligible count get position
 *     -1 and score NaN.  H <= 16384 when hist_article is given. */
size_t nrm_pool_workspace_bytes(int B, int H, int N, int chunk);
int nrm_forward_pool(const nrm_compact_batch* users, int B, int H, int N, int chunk, const float* params, const float* bn_running_mean,
                     const float* bn_running_var, int precision, float* logits, void* workspace, size_t workspace_bytes, void* stream);
int nrm_pool_topk(const float* logits, int n_models, long long model_stride, int B, int N, int k, const int* pool_article, int n_articles,
                  const int* hist_article, int H, int* pos_out, float* val_out, void* stream);

/* ---- UserModel.loss (user_model.py:37-43) ---------------------------------------- */
/* loss = (1-alpha) BCE(softmax(out), y) + alpha BCE(softmax(out + delta[id]), y), mean
 * over B*C, log clamped at -100 (nn.BCELoss).  Writes *loss (float32) and keeps the unit
 * gradients in `scratch` (>= nrm_loss_scratch_bytes(B,C)).  `scratch` must be ZERO-FILLED ONCE
 * before its first use (it holds the arrival counter with which the last block of the forward
 * kernel adds the block sums in fixed order; every call leaves the counter at zero again).
 * delta has delta_numel = user_num + 1 entries (user_model.py:23).  A user id outside [0, delta_numel) makes the reference
 * raise IndexError; here the loss of that step is NaN (no host synchronisation) and the backward ignores the id. */
size_t nrm_loss_scratch_bytes(int B, int C);
int nrm_loss_forward(const float* logits, const float* delta, long long delta_numel,
                     const long long* user_id, const double* label, int B, int C, float alpha,
                     float* loss, void* scratch, size_t scratch_bytes, void* stream);
/* grad_loss: device scalar dL/dloss.  dlogits [B,C]; ddelta: dense [delta_numel],
 * overwritten (zeros + per-user sums, duplicates combined in batch order). */
int nrm_loss_backward(const long long* user_id, int B, int C, const float* grad_loss,
                      float* dlogits, float* ddelta, long long delta_numel,
                      const void* scratch, size_t scratch_bytes, void* stream);

/* ---- torch.optim.Adam single step, coupled L2 (train.py:48,74) -------------------- */
/* g' = g + wd p; m = lerp(m, g', 1-b1); v = b2 v + (1-b2) g'^2;
 * p -= (lr / (1-b1^step)) * m / (sqrt(v)/sqrt(1-b2^step) + eps).  n floats, in place.
 * grad_scale multiplies g first (1/world_size for a summed data-parallel gradient). */
int nrm_adam_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, long long n,
                  float lr, float beta1, float beta2, float eps, float weight_decay,
                  long long step, float grad_scale, void* stream);

/* Same update with the hyper-parameters and the step counter on the device, so that a whole
 * training step can be captured in a CUDA graph and replayed: adam_state points to
 * { int64 step; float lr, beta1, beta2, eps, weight_decay, grad_scale, step_size, bc2_sqrt; }
 * (40 bytes).  Each call increments `step` and derives the bias corrections on the device. */
int nrm_adam_step_device(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, long long n,
                         void* adam_state, void* stream);

/* ---- batched ranking metrics (tool/evaluation.py:3-5, train.py:77-80, verify.py:25-37) ----- */
/* One result per impression b over its first n_valid[b] candidates (n_valid null = all C):
 *   auc[b]  sklearn.metrics.roc_auc_score(label, score) (ties averaged; NaN if one class is missing),
 *   hit[b]  argmax(score) == argmax(label)  (verify.py:32),
 *   rr[b]   reciprocal rank of the best-ranked positive (stable descending order, test.py:124-127),
 *   ndcg[b] nDCG@k with binary gains.   Any output pointer may be null.  scores: float32 [B, score_stride],
 * labels: float64 [B, label_stride] (label > 0.5 = clicked).  MRR / nDCG are not in the reference (unpinned). */
int nrm_batch_metrics(const float* scores, long long score_stride, const double* labels, long long label_stride,
                      const int* n_valid, int B, int C, int k, float* auc, float* hit, float* rr, float* ndcg,
                      void* stream);

/* ---- scoring epilogue and submission text (test.py:58-70, test.py:118-132) ------------------ */
/* logits: n_models stacked eval-mode outputs, model m / impression b at logits + m*model_stride + b*row_stride,
 * C float32 each (C = the batch's candidate columns after test.py:52-56 trimmed the common pad tail).
 * empty_num[b] (int64, device, may be null = 0) = pad candidates still at the end of row b.
 *   scores[b][i] = mean_m softmax(logits_m[b])[i]                       (softmax over all C columns, test.py:58-63)
 *                  then softmax over the first C - empty_num[b] entries again when empty_num[b] > 0 (test.py:65-68);
 *                  pad entries are written as 0.
 *   ranks[b][i]  = 1-based position of candidate i in the stable descending order of scores[b][0 : C - empty_num[b]]
 *                  (Python sorted(..., reverse=True), test.py:124-127); -1 for pad entries.  May be null.
 * scores: float32 [B, C], ranks: int32 [B, C]. */
int nrm_score_epilogue(const float* logits, int n_models, long long model_stride, long long row_stride, int B, int C,
                       const long long* empty_num, float* scores, int* ranks, void* stream);

/* Text of test.py:129-130 for a whole batch: line b = "{impression_id[b]} [{ranks[b][0]},{ranks[b][1]},...]\n" over the
 * non-pad candidates.  offsets: int64 [B + 1] (device) receives the byte offset of every line, offsets[B] = total
 * length; out: at least `capacity` bytes (nrm_rank_strings_capacity(B, C) is always enough).  Lines that would end
 * beyond `capacity` are not written (offsets[B] > capacity tells the caller). */
size_t nrm_rank_strings_capacity(int B, int C);
int nrm_rank_strings(const long long* impression_id, const int* ranks, const long long* empty_num, int B, int C,
                     long long* offsets, char* out, long long capacity, void* stream);

/* ---- compact wire format (additional entry point; tool/process_data.py:195-252 defines the packed one) -------- */
/* Rebuilds the reference's packed float64 inputs in device memory from an article table and per-impression ids:
 *   articles     float32 [n_articles, 80]: pca 64 | category | sub-category 5 | sentiment 3 | type | total_inviews,
 *                total_pageviews, total_read_time | 3 pad floats; row 0 all-zero = the pad article (ids out of range read it)
 *   hist_article int32 [B,H];  hist_time uint32 [B,H] = years | months << 12 | days << 16 | hours << 21
 *                (the four integers of tool/normalization.py:31-39);  hist_click float32 [B,H,2] = read_time, scroll
 *   cand_article int32 [B,C];  cand_time uint32 [B,C];  label32 float32 [B,C] (may be null)
 * Outputs (all contiguous, 16-byte aligned): x_history float64 [B,H,80], x_target float64 [B,C,78], x_global float64
 * [B,C,3], label64 float64 [B,C] (when label32 is given).  The model reads its inputs as float32
 * (user_invariant_interest_model.py:74-75), so nrm_forward on these tensors equals nrm_forward on the ETL's own. */
int nrm_expand_compact(const float* articles, int n_articles, const int* hist_article, const unsigned* hist_time,
                       const float* hist_click, const int* cand_article, const unsigned* cand_time, const float* label32,
                       int B, int H, int C, double* x_history, double* x_target, double* x_global, double* label64,
                       void* stream);

#ifdef __cplusplus
}
#endif
#endif /* NRM_B200_H */
