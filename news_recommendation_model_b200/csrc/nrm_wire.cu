// Compact wire format ("next" row N3 of SURVEY.md section 8f).
// The reference ETL (tool/process_data.py:195-252) materialises every impression as float64 rows that repeat the whole
// article record for every click and every candidate: 640 B per history row, 624 + 24 B per candidate, ids stored as
// doubles.  Only 6 of those 80 numbers belong to the click (4 time buckets, read time, scroll); the other 74 (+ the 3
// "global" article statistics of x_global) are a function of the article.  The compact format keeps
//     articles     [n_articles, 80] float32   pca 64 | category | sub-category 5 | sentiment 3 | type | inviews, pageviews,
//                                             read_time | 3 pad;  row 0 is all-zero (the pad article)
// resident in HBM and sends per impression
//     hist_article [B,H] int32, hist_time [B,H] uint32 (years | months << 12 | days << 16 | hours << 21, the integers of
//     tool/normalization.py:31-39), hist_click [B,H,2] float32 (read_time, scroll)           -> 16 B per history row
//     cand_article [B,C] int32, cand_time [B,C] uint32                                       ->  8 B per candidate
//     label [B,C] float32
// The model consumes x.to(torch.float32) (user_invariant_interest_model.py:74-75), so float32 storage loses nothing.
// expand_compact_kernel rebuilds the reference's packed float64 tensors in HBM (one warp per row: 320 B gathered,
// 640 B written, all 16-byte accesses), after which the unchanged forward / backward kernels run; results are bit for
// bit those of feeding the packed tensors.
#include "nrm_kernels.cuh"

namespace nrm {

constexpr int ART_COLS = 80;        // floats per article row
constexpr int ART_G = 74;           // first of the three global statistics

__global__ void __launch_bounds__(256)
expand_compact_kernel(const float* __restrict__ articles, int n_articles,
                      const int* __restrict__ hist_article, const unsigned* __restrict__ hist_time, const float* __restrict__ hist_click,
                      const int* __restrict__ cand_article, const unsigned* __restrict__ cand_time, const float* __restrict__ label32,
                      long long NH, long long R, double* __restrict__ xh, double* __restrict__ xt, double* __restrict__ xg,
                      double* __restrict__ label64) {
  const long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= NH + R) {                                        // tail warps: label float32 -> float64
    const long long i = (row - NH - R) * 32 + lane;
    if (label32 != nullptr && i < R) label64[i] = (double)label32[i];
    return;
  }
  const bool is_hist = row < NH;
  const long long r = is_hist ? row : row - NH;
  int art = is_hist ? hist_article[r] : cand_article[r];
  art = (art < 0 || art >= n_articles) ? 0 : art;             // out-of-range ids read the pad article
  double* dst = is_hist ? xh + r * HC : xt + r * TC;
  if (lane < 20) {
    const float4 v = __ldg(reinterpret_cast<const float4*>(articles + (long long)art * ART_COLS) + lane);
    if (lane < 18) {                                          // article columns 4 lane .. 4 lane + 3 -> packed columns 4 + ...
      double2* d = reinterpret_cast<double2*>(dst + 4 + 4 * lane);
      d[0] = make_double2((double)v.x, (double)v.y);
      d[1] = make_double2((double)v.z, (double)v.w);
    } else if (lane == 18) {                                  // sentiment[2], type | inviews, pageviews
      *reinterpret_cast<double2*>(dst + 76) = make_double2((double)v.x, (double)v.y);
      if (!is_hist) { xg[r * GC + 0] = (double)v.z; xg[r * GC + 1] = (double)v.w; }
    } else if (!is_hist) {                                    // read_time statistic
      xg[r * GC + 2] = (double)v.x;
    }
  } else if (lane == 20) {
    const unsigned t = is_hist ? hist_time[r] : cand_time[r];
    double2* d = reinterpret_cast<double2*>(dst);
    d[0] = make_double2((double)(t & 0xfffu), (double)((t >> 12) & 0xfu));
    d[1] = make_double2((double)((t >> 16) & 0x1fu), (double)((t >> 21) & 0x1fu));
  } else if (lane == 21 && is_hist) {
    const float2 c = __ldg(reinterpret_cast<const float2*>(hist_click) + r);
    *reinterpret_cast<double2*>(dst + 78) = make_double2((double)c.x, (double)c.y);
  }
}

int launch_expand_compact(const float* articles, int n_articles, const int* hist_article, const unsigned* hist_time, const float* hist_click,
                          const int* cand_article, const unsigned* cand_time, const float* label32, long long NH, long long R,
                          double* x_history, double* x_target, double* x_global, double* label64, cudaStream_t s) {
  const long long warps = NH + R + (R + 31) / 32;
  expand_compact_kernel<<<(unsigned)((warps + 7) / 8), 256, 0, s>>>(articles, n_articles, hist_article, hist_time, hist_click, cand_article,
                                                                    cand_time, label32, NH, R, x_history, x_target, x_global, label64);
  NRM_LAUNCH_CHECK("expand_compact_kernel");
  return NRM_OK;
}

}  // namespace nrm

using namespace nrm;

extern "C" int nrm_expand_compact(const float* articles, int n_articles, const int* hist_article, const unsigned* hist_time,
                                  const float* hist_click, const int* cand_article, const unsigned* cand_time, const float* label32,
                                  int B, int H, int C, double* x_history, double* x_target, double* x_global, double* label64,
                                  void* stream) {
  if (!articles || n_articles <= 0 || !hist_article || !hist_time || !hist_click || !cand_article || !cand_time || B <= 0 || H <= 0 ||
      C <= 0 || !x_history || !x_target || !x_global || (label32 && !label64)) {
    set_error("nrm_expand_compact: bad argument"); return NRM_EINVAL;
  }
  if ((reinterpret_cast<uintptr_t>(articles) | reinterpret_cast<uintptr_t>(x_history) | reinterpret_cast<uintptr_t>(x_target)) & 15) {
    set_error("nrm_expand_compact: articles / x_history / x_target must be 16-byte aligned"); return NRM_EINVAL;
  }
  return launch_expand_compact(articles, n_articles, hist_article, hist_time, hist_click, cand_article, cand_time, label32, (long long)B * H,
                               (long long)B * C, x_history, x_target, x_global, label64, (cudaStream_t)stream);
}
