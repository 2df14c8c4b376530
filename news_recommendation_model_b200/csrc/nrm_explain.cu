// "Why this article": the k history clicks with the largest attention scores per (branch, impression, candidate).
// Input: the [2,B,C,H] scores nrm_forward_scores exports (s_label, s_ti of user_invariant_interest_model.py:83-87).  Output: the
// k best history positions per row and their scores, in the stable descending order of Python's sorted(..., reverse=True) that
// test.py:124-127 uses for candidates (ties go to the lower history index).  Pad rows (all-zero packed history rows,
// tool/process_data.py:198, or article id 0 in the compact format) never appear; slots beyond an impression's real clicks get
// index -1 and score NaN.
//
// One CTA per impression: its pad mask is built once in shared memory (all threads, coalesced 16-byte loads of the packed rows) and
// shared by the 2C rows, which the CTA's warps (up to TOPK_WARPS_MAX, fewer when H is too long for their keys) take in turn.  A
// row's keys (order-preserving score bits << 32 | ~h; 0 = pad or taken) sit in shared memory, each lane owning the positions
// h = lane (mod 32) and caching its own best key; a round is one warp max, after which only the winning lane rescans.
#include "nrm_kernels.cuh"

namespace nrm {

constexpr int TOPK_WARPS_MAX = 16;
constexpr int TOPK_MAX = 64;

// (score, h) -> a key whose unsigned order is the stable descending order; -0.0 and +0.0 are equal, as Python compares them
__device__ __forceinline__ unsigned long long topk_key(float v, int h) {
  unsigned u = __float_as_uint(v + 0.0f);
  u = (u & 0x80000000u) ? ~u : (u | 0x80000000u);
  return ((unsigned long long)u << 32) | (unsigned)~h;      // ~h > 0 for every h >= 0: a real row never has key 0
}

__global__ void __launch_bounds__(TOPK_WARPS_MAX * 32, 1)
history_topk_kernel(const float* __restrict__ scores, int B, int C, int H, int k, const double* __restrict__ x_history,
                    const int* __restrict__ hist_article, int* __restrict__ idx_out, float* __restrict__ val_out) {
  extern __shared__ __align__(16) unsigned char topk_smem[];
  const int nwarps = blockDim.x >> 5, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  unsigned long long* keys = reinterpret_cast<unsigned long long*>(topk_smem) + (size_t)warp * H;   // [nwarps][H]
  unsigned char* real = topk_smem + (size_t)nwarps * H * 8;                                          // [H]: 1 = a click, 0 = pad row
  for (int b = blockIdx.x; b < B; b += gridDim.x) {
    __syncthreads();                                         // the previous impression's mask is no longer read
    for (int h = threadIdx.x; h < H; h += blockDim.x)
      real[h] = x_history != nullptr ? 0 : hist_article == nullptr ? 1 : hist_article[(long long)b * H + h] != 0;
    if (x_history != nullptr) {                              // an all-zero packed row of 80 float64 is padding
      __syncthreads();
      const double2* rows = reinterpret_cast<const double2*>(x_history + (long long)b * H * HC);
      for (int i = threadIdx.x; i < H * (HC / 2); i += blockDim.x) {
        const double2 v = rows[i];
        if (v.x != 0.0 || v.y != 0.0) real[i / (HC / 2)] = 1;
      }
    }
    __syncthreads();
    for (int r = warp; r < 2 * C; r += nwarps) {
      const int branch = r >= C ? 1 : 0, c = r - branch * C;
      const long long row = ((long long)branch * B + b) * C + c;
      const float* s = scores + row * H;
      unsigned long long best = 0;
      for (int h = lane; h < H; h += 32) {
        const unsigned long long key = real[h] ? topk_key(s[h], h) : 0ull;
        keys[h] = key;
        best = key > best ? key : best;
      }
      for (int j = 0; j < k; ++j) {
        unsigned long long m = best;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          const unsigned long long other = __shfl_xor_sync(0xffffffffu, m, o);
          m = other > m ? other : m;
        }
        const int h = m != 0 ? (int)~(unsigned)m : -1;
        if (lane == (j & 31)) {
          idx_out[row * k + j] = h;
          val_out[row * k + j] = h >= 0 ? s[h] : __int_as_float(0x7fc00000);
        }
        if (h >= 0 && (h & 31) == lane) {                    // the winner's owner takes it out and finds its next best
          keys[h] = 0ull;
          best = 0;
          for (int i = lane; i < H; i += 32) best = keys[i] > best ? keys[i] : best;
        }
      }
    }
  }
}


}  // namespace nrm

using namespace nrm;

extern "C" int nrm_history_topk(const float* scores, int B, int C, int H, int k, const double* x_history, const int* hist_article,
                                int* idx_out, float* val_out, void* stream) {
  if (!scores || !idx_out || !val_out) { set_error("nrm_history_topk: null pointer"); return NRM_EINVAL; }
  if (B <= 0 || C <= 0 || H <= 0) { set_error("nrm_history_topk: B, C, H must be positive (got %d, %d, %d)", B, C, H); return NRM_EINVAL; }
  if (k < 1 || k > H || k > TOPK_MAX) { set_error("nrm_history_topk: need 1 <= k <= min(H, %d) (got k = %d, H = %d)", TOPK_MAX, k, H); return NRM_EINVAL; }
  if (x_history && hist_article) { set_error("nrm_history_topk: pass at most one of x_history / hist_article"); return NRM_EINVAL; }
  int dev = 0, smem_max = 0;
  NRM_CUDA(cudaGetDevice(&dev));
  NRM_CUDA(cudaDeviceGetAttribute(&smem_max, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
  const long long per_warp = 8LL * H;                      // a row's keys; + H bytes of pad mask per CTA
  const int nwarps = (int)min((long long)TOPK_WARPS_MAX, ((long long)smem_max - H) / per_warp);
  if (nwarps < 1) { set_error("nrm_history_topk: H = %d does not fit the %d bytes of shared memory of a CTA", H, smem_max); return NRM_EINVAL; }
  const size_t smem = (size_t)(nwarps * per_warp + H);
  NRM_CUDA(cudaFuncSetAttribute(history_topk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  history_topk_kernel<<<B, nwarps * 32, smem, (cudaStream_t)stream>>>(scores, B, C, H, k, x_history, hist_article, idx_out, val_out);
  NRM_LAUNCH_CHECK("history_topk_kernel");
  return NRM_OK;
}
