// Internal launcher interface between the translation units of libnrm_b200.
#pragma once
#include "nrm_common.cuh"

namespace nrm {

// compact wire format (nrm_wire.cu): the article table resident in HBM + per-impression ids / time buckets / click features
struct CompactPtrs {
  const float* articles; int n_articles;     // [n,80] float32: pca 64 | category | sub-category 5 | sentiment 3 | type | 3 global statistics | pad
  const int* hist_article; const unsigned* hist_time; const float* hist_click;   // [B,H], [B,H], [B,H,2]
  const int* cand_article; const unsigned* cand_time;                            // [B,C], [B,C]
  const float* label32; double* label64;     // optional: float32 labels -> the float64 labels the loss kernels read
};
struct BatchPtrs {
  const double* xh;               // [B,H,80]
  const double* xt; long long xt_bs;   // [B,C,78], batch stride in doubles
  const double* xg; long long xg_bs;   // [B,C,3]
  const CompactPtrs* compact = nullptr;   // non-null: the packed pointers above are unused, the row kernels read the compact format
};

// nrm_embed.cu
int launch_embed_rows(const BatchPtrs& in, const float* P, Workspace& w, bool with_keys, cudaStream_t s);
int launch_table_sort(Workspace& w, cudaStream_t s);                  // counting sort of the table ids (needs only the forward's keys)
int launch_table_grads(Workspace& w, float* grads, cudaStream_t s);  // segmented sums -> table gradients (after launch_table_sort)
int launch_small_linear_grads(const BatchPtrs& in, Workspace& w, float* grads, cudaStream_t s);

// nrm_w1.cu
int launch_w1_forward(const float* P, Workspace& w, cudaStream_t s);             // w.xin_h -> w.xh
int launch_w1_backward(const float* P, Workspace& w, float* grads, cudaStream_t s);  // w.dxh -> w.dxin_h, w1 gradients

// nrm_w1_tc.cu  (tensor-core tiles; precision = bf16 / bf16x3)
int launch_w1_forward_tc(const float* P, Workspace& w, int precision, cudaStream_t s);
int launch_w1_backward_tc(const float* P, Workspace& w, float* grads, int precision, cudaStream_t s);

// nrm_attention.cu  (branch 0 = label attention on w1-projected features, 1 = text/img PCA)
int launch_attention_forward(const BatchPtrs& in, const float* P, Workspace& w, int branch, int precision, cudaStream_t s);
int launch_attention_backward(const BatchPtrs& in, const float* P, Workspace& w, int branch, int precision, cudaStream_t s);
int launch_attention_finish(const float* P, Workspace& w, int branch, int precision, float* grads, cudaStream_t s);

// nrm_attention_tc.cu  (precision = bf16 / bf16x3: tcgen05 tensor-core tiles)
int launch_attention_prep(const float* P, Workspace& w, cudaStream_t s);          // derived weights -> w.att_derived (weights only)
int launch_candidate_tp(const float* P, Workspace& w, cudaStream_t s);            // per-candidate tp -> w.tp (needs w.e target rows)
int launch_attention_forward_tc(const BatchPtrs& in, Workspace& w, int branch, int precision, cudaStream_t s);
int launch_attention_backward_tc(const BatchPtrs& in, const float* P, Workspace& w, int branch, int precision, cudaStream_t s);
int launch_attention_finish_tc(const float* P, Workspace& w, float* grads, cudaStream_t s);   // both branches

// nrm_attention_rs.cu  (row-stacked M = 128 formulation, operand rows in tensor memory; precision = bf16 / bf16x3)
size_t attention_rs_image_bytes();
int rsprof_read(long long* host_out64);                                         // -DNRM_RS_PROFILE builds only
int launch_attention_prep_rs(const float* P, Workspace& w, cudaStream_t s);       // weight image -> w.att_rs_img (weights only)
int launch_attention_forward_rs(const BatchPtrs& in, Workspace& w, int precision, cudaStream_t s);   // both branches, one launch
int launch_attention_forward_rs_scores(Workspace& w, int precision, cudaStream_t s);   // the same + scores to w.scores (nrm_attention_rs_scores.cu)
// nrm_attention_rs_bwd.cu: sums over rows (weight gradients, dtp) of one branch; export_dhid also writes the dhid tiles / scores
int launch_attention_backward_rs(Workspace& w, int branch, int precision, bool export_dhid, cudaStream_t s);
int launch_attention_input_grad_rs(Workspace& w, int precision, cudaStream_t s);   // label branch: dxh, dxt from the exported tiles
long long attention_rs_tiles(int B, int H, int C);
bool use_rowstacked();

// nrm_head_fused.cu
int launch_head_transpose(const float* P, Workspace& w, cudaStream_t s);          // transposed head matrices -> w.head_wt (weights only)
int launch_head_forward_fused(const float* P, Workspace& w, float* run_mean, float* run_var, long long* nbt, int training, int keep,
                              const double* bn_sums, long long bn_rows, float* logits, cudaStream_t s);
int launch_head_backward_dgrad(const float* P, Workspace& w, const float* dlogits, cudaStream_t s);
int launch_head_backward_bn(Workspace& w, float* grads, cudaStream_t s, int dgrad_tiles);   // dgrad_tiles: row tiles of the dgrad kernel (0 = FFMA kernel's)                   // -> w.bn_bwd_sums, bn.weight / bn.bias gradients
int launch_head_backward_wgrad(const float* P, Workspace& w, float* grads, cudaStream_t s, int dgrad_tiles, int tc_precision = 0);   // tc_precision != 0: products on tcgen05   // weight gradients of the five Linear layers + out_mlp.fc2
int launch_head_backward_fused(const float* P, Workspace& w, const float* dlogits, float* grads, cudaStream_t s);   // -> w.bn_bwd_sums, w.dz, w.de

// nrm_head_tc.cu  (tensor-core head; precision = bf16 / bf16x3)
size_t head_tc_image_bytes();
int headprof_read(long long* host_out32);                                       // -DNRM_RS_PROFILE builds only
int launch_head_images_tc(const float* P, Workspace& w, int precision, bool with_backward, cudaStream_t s);   // weights only -> w.head_img
int head_tc_tiles(long long R);
int launch_head_wgrad_tc(const float* P, Workspace& w, int precision, int rows_per_chunk, int nchunks, cudaStream_t s);   // partials in head_wgrad_kernel's layout
// tensor-core data-gradient chain: as launch_head_backward_dgrad + launch_head_backward_bn, except that w.de holds dx (not dx * gate)
int launch_head_backward_dgrad_tc(const float* P, Workspace& w, int precision, const float* dlogits, float* grads, cudaStream_t s);
int launch_head_forward_tc(const float* P, Workspace& w, int precision, float* run_mean, float* run_var, long long* nbt, int training, int keep,
                           const double* bn_sums, long long bn_rows, float* logits, cudaStream_t s);

// nrm_head.cu
int launch_bn_partial_sums(Workspace& w, cudaStream_t s);                 // -> w.bn_sums
int launch_head_forward(const float* P, Workspace& w, float* run_mean, float* run_var, long long* nbt,
                        int training, int keep, const double* bn_sums, long long global_rows, float* logits, cudaStream_t s);
int launch_head_backward(const float* P, Workspace& w, const float* dlogits, float* grads, cudaStream_t s);  // -> w.bn_bwd_sums
int launch_bn_backward_combine(const float* P, Workspace& w, int training, const double* bn_bwd_sums,
                               long long global_rows, bool de_holds_dx, cudaStream_t s);  // w.de += BN path

}  // namespace nrm
