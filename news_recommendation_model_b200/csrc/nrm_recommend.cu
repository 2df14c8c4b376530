// Recommendation from a shared article pool: per user, the k eligible pool positions with the largest score (nrm_pool_topk).
// Input: the [M][B][N] logits nrm_forward_pool computed for every (user, pool article) pair, one slice per model of an ensemble.
// A position is eligible unless its article id is 0 or outside [1, n_articles), one of its logits is NaN, or (hist_article given)
// the user has already clicked that article.  The score is the logit (M = 1) or the mean over the models of the softmax over
// the user's eligible positions (M >= 2, test.py:58-63).  Output order is Python's stable sorted(..., reverse=True)
// (test.py:124-127): descending score, ties to the lower position; slots beyond the eligible count get position -1, score NaN.
//
// One CTA of POOL_THREADS per user.  The user's clicked ids go into an open-addressing hash table in shared memory once.  Every
// pass over the pool recomputes a position's order-preserving 64-bit key (score bits << 32 | ~position; 0 = not eligible) from
// the logits, so no workspace is needed: M >= 2 first takes the per-model masked max and sum-exp with block reductions, then a
// radix select over the keys (11-bit digits, most significant first) finds the k-th largest key, usually in 2-3 passes since
// the search stops as soon as the chosen digit's bucket holds exactly the keys still missing.  A last pass gathers the <= k keys
// at or above it into shared memory, where a bitonic sort orders them.  Keys are unique, so the selection and its order are
// exact; every sum is taken in a fixed order, so results do not depend on timing.
#include <math_constants.h>

#include "nrm_kernels.cuh"

namespace nrm {

constexpr int POOL_THREADS = 512;
constexpr int POOL_TOPK_MAX = 1024;
constexpr int POOL_MODELS_MAX = 16;
constexpr int POOL_HASH_LG_MAX = 15;          // 32768 slots (128 KB): up to 16384 history rows per user
constexpr int RADIX_BITS = 11, RADIX_BINS = 1 << RADIX_BITS;

struct PoolTopkArgs {
  const float* logits; int n_models; long long model_stride;
  int N, k;
  const int* pool_article; int n_articles;
  const int* hist_article; int H; int hash_lg;   // hash_lg 0: no exclusion
  int* pos_out; float* val_out;
};

// (score, position) -> a key whose unsigned order is the stable descending order (as nrm_explain.cu's; -0.0 == +0.0)
__device__ __forceinline__ unsigned long long pool_key(float v, int n) {
  unsigned u = __float_as_uint(v + 0.0f);
  u = (u & 0x80000000u) ? ~u : (u | 0x80000000u);
  return ((unsigned long long)u << 32) | (unsigned)~n;
}
__device__ __forceinline__ float pool_key_score(unsigned long long key) {
  const unsigned u = (unsigned)(key >> 32);
  return __uint_as_float((u & 0x80000000u) ? (u & 0x7fffffffu) : ~u);
}

__device__ __forceinline__ unsigned pool_hash(int id, int lg) { return ((unsigned)id * 0x9E3779B1u) >> (32 - lg); }

__device__ __forceinline__ bool pool_clicked(const int* tab, int lg, int id) {
  if (lg == 0) return false;
  const unsigned m = (1u << lg) - 1;
  for (unsigned h = pool_hash(id, lg);; h = (h + 1) & m) {     // load factor <= 1/2: an empty slot ends every probe
    const int v = tab[h];
    if (v == id) return true;
    if (v == 0) return false;
  }
}

// Every pass walks the pool in steps of POOL_BATCH positions per thread (n0 + j * POOL_THREADS), loading all of them before using
// any, so that a thread keeps POOL_BATCH independent loads in flight.
constexpr int POOL_BATCH = 4;

// a pool id that may be recommended: in range and not clicked by this user
__device__ __forceinline__ bool pool_id_ok(const PoolTopkArgs& a, const int* tab, int id) {
  return id >= 1 && id < a.n_articles && !pool_clicked(tab, a.hash_lg, id);
}

// keys of positions n0 + j * POOL_THREADS from the logits alone (0: past the pool or a NaN logit in some model) and their ids;
// whether the id is eligible is left to the caller, which checks it only for the keys it wants
template <bool ENSEMBLE>
__device__ __forceinline__ void pool_raw_keys(const PoolTopkArgs& a, const float* row, const float* mx, const float* sum, int n0,
                                              unsigned long long (&key)[POOL_BATCH], int (&id)[POOL_BATCH]) {
  float x[POOL_BATCH], acc[POOL_BATCH];
  bool ok[POOL_BATCH];
#pragma unroll
  for (int j = 0; j < POOL_BATCH; ++j) {
    const int n = n0 + j * POOL_THREADS;
    ok[j] = n < a.N;
    id[j] = ok[j] ? __ldg(a.pool_article + n) : 0;
    x[j] = ok[j] ? row[n] : 0.f;
  }
#pragma unroll
  for (int j = 0; j < POOL_BATCH; ++j) {
    ok[j] = ok[j] && x[j] == x[j];
    if (ENSEMBLE) acc[j] = expf(x[j] - mx[0]) / sum[0];
  }
  if (ENSEMBLE) {
    for (int m = 1; m < a.n_models; ++m) {
      const float* xm = row + (long long)m * a.model_stride;
#pragma unroll
      for (int j = 0; j < POOL_BATCH; ++j) x[j] = n0 + j * POOL_THREADS < a.N ? xm[n0 + j * POOL_THREADS] : 0.f;
#pragma unroll
      for (int j = 0; j < POOL_BATCH; ++j) {
        ok[j] = ok[j] && x[j] == x[j];
        acc[j] += expf(x[j] - mx[m]) / sum[m];
      }
    }
  }
#pragma unroll
  for (int j = 0; j < POOL_BATCH; ++j) key[j] = ok[j] ? pool_key(ENSEMBLE ? acc[j] / (float)a.n_models : x[j], n0 + j * POOL_THREADS) : 0ull;
}

// ensemble statistics: this thread's max (MAX) or sum of exp(x_m - vmax) over its eligible positions, for model m
template <bool MAX>
__device__ __forceinline__ float pool_model_partial(const PoolTopkArgs& a, const float* row, const int* tab, int m, float vmax) {
  float v = MAX ? -CUDART_INF_F : 0.f;
#pragma unroll 1
  for (int n0 = threadIdx.x; n0 < a.N; n0 += POOL_BATCH * POOL_THREADS) {
    int id[POOL_BATCH];
    float xm[POOL_BATCH];
    bool ok[POOL_BATCH];
#pragma unroll
    for (int j = 0; j < POOL_BATCH; ++j) {
      const int n = n0 + j * POOL_THREADS;
      ok[j] = n < a.N;
      id[j] = ok[j] ? __ldg(a.pool_article + n) : 0;
      xm[j] = ok[j] ? row[(long long)m * a.model_stride + n] : 0.f;
    }
    for (int mm = 0; mm < a.n_models; ++mm) {            // a NaN in any model makes the position ineligible for all of them
      float x[POOL_BATCH];
#pragma unroll
      for (int j = 0; j < POOL_BATCH; ++j) x[j] = ok[j] ? row[(long long)mm * a.model_stride + n0 + j * POOL_THREADS] : 0.f;
#pragma unroll
      for (int j = 0; j < POOL_BATCH; ++j) ok[j] = ok[j] && x[j] == x[j];
    }
#pragma unroll
    for (int j = 0; j < POOL_BATCH; ++j)
      if (ok[j] && pool_id_ok(a, tab, id[j])) v = MAX ? fmaxf(v, xm[j]) : v + expf(xm[j] - vmax);
  }
  return v;
}

// block reduction in a fixed order (warp butterflies, then warp 0 over the warp results); every thread gets the result
template <bool MAX>
__device__ __forceinline__ float pool_block_reduce(float v, float* red) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float w = __shfl_xor_sync(0xffffffffu, v, o);
    v = MAX ? fmaxf(v, w) : v + w;
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  __syncthreads();                                         // red[] of a previous reduction has been read
  if (lane == 0) red[warp] = v;
  __syncthreads();
  if (warp == 0) {
    v = lane < POOL_THREADS / 32 ? red[lane] : (MAX ? -CUDART_INF_F : 0.f);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float w = __shfl_xor_sync(0xffffffffu, v, o);
      v = MAX ? fmaxf(v, w) : v + w;
    }
    if (lane == 0) red[POOL_THREADS / 32] = v;
  }
  __syncthreads();
  return red[POOL_THREADS / 32];
}

template <bool ENSEMBLE>
__global__ void __launch_bounds__(POOL_THREADS, 3)
pool_topk_kernel(const PoolTopkArgs a) {
  extern __shared__ int clicked_tab[];                     // [1 << hash_lg] article ids, 0 = empty slot
  __shared__ unsigned hist[RADIX_BINS];
  __shared__ unsigned long long sel[POOL_TOPK_MAX];
  __shared__ float red[POOL_THREADS / 32 + 1];
  __shared__ float mx[POOL_MODELS_MAX], sum[POOL_MODELS_MAX];
  __shared__ unsigned long long s_prefix;
  __shared__ unsigned s_need, s_done, s_count;
  const int tid = threadIdx.x, b = blockIdx.x, N = a.N;
  const float* row = a.logits + (long long)b * N;

  // the user's clicked ids (pad rows and ids no pool position can carry are left out)
  if (a.hash_lg > 0) {
    const int cap = 1 << a.hash_lg;
    for (int i = tid; i < cap; i += POOL_THREADS) clicked_tab[i] = 0;
    __syncthreads();
    for (int h = tid; h < a.H; h += POOL_THREADS) {
      const int id = a.hist_article[(long long)b * a.H + h];
      if (id < 1 || id >= a.n_articles) continue;
      for (unsigned s = pool_hash(id, a.hash_lg);; s = (s + 1) & (unsigned)(cap - 1)) {
        const int old = atomicCAS(&clicked_tab[s], 0, id);
        if (old == 0 || old == id) break;
      }
    }
  }
  __syncthreads();

  // ensemble: per model, max and sum of exp(x - max) over the eligible positions
  if (ENSEMBLE) {
    for (int m = 0; m < a.n_models; ++m) {
      const float vmax = pool_block_reduce<true>(pool_model_partial<true>(a, row, clicked_tab, m, 0.f), red);
      const float vsum = pool_block_reduce<false>(pool_model_partial<false>(a, row, clicked_tab, m, vmax), red);
      if (tid == 0) { mx[m] = vmax; sum[m] = vsum; }
    }
    __syncthreads();
  }

  // radix select of the k-th largest key; threshold: the selected keys are exactly those >= it
  unsigned long long prefix = 0ull, mask = 0ull, threshold = 0ull;
  unsigned need = (unsigned)a.k;
  for (int shift = 64 - RADIX_BITS;; shift = shift > RADIX_BITS ? shift - RADIX_BITS : 0) {
    for (int i = tid; i < RADIX_BINS; i += POOL_THREADS) hist[i] = 0;
    __syncthreads();
#pragma unroll 1
    for (int n0 = tid; n0 < N; n0 += POOL_BATCH * POOL_THREADS) {
      unsigned long long key[POOL_BATCH];
      int id[POOL_BATCH];
      pool_raw_keys<ENSEMBLE>(a, row, mx, sum, n0, key, id);
#pragma unroll
      for (int j = 0; j < POOL_BATCH; ++j)
        if (key[j] != 0ull && (key[j] & mask) == prefix && pool_id_ok(a, clicked_tab, id[j]))
          atomicAdd(&hist[(unsigned)(key[j] >> shift) & (RADIX_BINS - 1)], 1u);
    }
    __syncthreads();
    if (tid < 32) {                                        // warp 0: lane l owns bins [64 l, 64 l + 64)
      constexpr int PER = RADIX_BINS / 32;
      unsigned own = 0;
#pragma unroll 8
      for (int i = 0; i < PER; ++i) own += hist[tid * PER + i];
      unsigned suf = own;                                  // keys in the bins of lanes >= tid
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const unsigned v = __shfl_down_sync(0xffffffffu, suf, o);
        if (tid + o < 32) suf += v;
      }
      const unsigned total = __shfl_sync(0xffffffffu, suf, 0);
      if (mask == 0ull && total <= need) {                 // first pass: no more eligible positions than slots
        if (tid == 0) { s_prefix = 1ull; s_need = total; s_done = 2; }
      } else {
        const unsigned above = suf - own;
        if (above < need && need <= suf) {
          unsigned acc = above;
#pragma unroll 1
          for (int i = PER - 1; i >= 0; --i) {
            const unsigned c = hist[tid * PER + i];
            if (acc + c >= need) {
              const unsigned long long d = (unsigned long long)(tid * PER + i);
              s_prefix = (prefix & ~((unsigned long long)(RADIX_BINS - 1) << shift)) | (d << shift);
              s_need = need - acc;
              s_done = c == need - acc;
              break;
            }
            acc += c;
          }
        }
      }
    }
    __syncthreads();
    const unsigned done = s_done;
    if (done == 2) { threshold = 1ull; break; }
    prefix = s_prefix;
    mask |= (unsigned long long)(RADIX_BINS - 1) << shift;
    need = s_need;
    if (done) { threshold = prefix; break; }
    __syncthreads();                                       // s_* are rewritten by the next pass
  }

  // gather the selected keys, then sort them descending (bitonic, padded with 0 keys to a power of two)
  if (tid == 0) s_count = 0;
  __syncthreads();
#pragma unroll 1
  for (int n0 = tid; n0 < N; n0 += POOL_BATCH * POOL_THREADS) {
    unsigned long long key[POOL_BATCH];
    int id[POOL_BATCH];
    pool_raw_keys<ENSEMBLE>(a, row, mx, sum, n0, key, id);
#pragma unroll
    for (int j = 0; j < POOL_BATCH; ++j)
      if (key[j] != 0ull && key[j] >= threshold && pool_id_ok(a, clicked_tab, id[j])) sel[atomicAdd(&s_count, 1u)] = key[j];
  }
  __syncthreads();
  const int cnt = (int)s_count;
  int P = 1;
  while (P < cnt) P <<= 1;
  for (int i = cnt + tid; i < P; i += POOL_THREADS) sel[i] = 0ull;
  __syncthreads();
  for (int size = 2; size <= P; size <<= 1) {
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      for (int t = tid; t < P / 2; t += POOL_THREADS) {
        const int lo = 2 * t - (t & (stride - 1)), hi = lo + stride;
        const bool desc = (lo & size) == 0;
        const unsigned long long x = sel[lo], y = sel[hi];
        if ((x < y) == desc) { sel[lo] = y; sel[hi] = x; }
      }
      __syncthreads();
    }
  }
  for (int j = tid; j < a.k; j += POOL_THREADS) {
    const long long o = (long long)b * a.k + j;
    if (j < cnt) {
      const unsigned long long key = sel[j];
      a.pos_out[o] = (int)~(unsigned)key;
      a.val_out[o] = pool_key_score(key);
    } else {
      a.pos_out[o] = -1;
      a.val_out[o] = CUDART_NAN_F;
    }
  }
}

int launch_pool_topk(const float* logits, int n_models, long long model_stride, int B, int N, int k, const int* pool_article, int n_articles,
                     const int* hist_article, int H, int* pos_out, float* val_out, cudaStream_t s) {
  if (k < 1 || k > N || k > POOL_TOPK_MAX) { set_error("nrm_pool_topk: need 1 <= k <= min(N, %d) (got k = %d, N = %d)", POOL_TOPK_MAX, k, N); return NRM_EINVAL; }
  if (n_models < 1 || n_models > POOL_MODELS_MAX) { set_error("nrm_pool_topk: need 1 <= n_models <= %d (got %d)", POOL_MODELS_MAX, n_models); return NRM_EINVAL; }
  if (n_models > 1 && model_stride < (long long)B * N) { set_error("nrm_pool_topk: model_stride smaller than B * N"); return NRM_EINVAL; }
  int lg = 0;
  if (hist_article != nullptr) {
    if (H <= 0) { set_error("nrm_pool_topk: H must be positive with hist_article (got %d)", H); return NRM_EINVAL; }
    lg = 5;
    while (lg <= POOL_HASH_LG_MAX && (1LL << lg) < 2LL * H) ++lg;
    if (lg > POOL_HASH_LG_MAX) { set_error("nrm_pool_topk: H = %d exceeds the %d history rows the exclusion table holds", H, 1 << (POOL_HASH_LG_MAX - 1)); return NRM_EINVAL; }
  }
  const PoolTopkArgs args{logits, n_models, model_stride, N, k, pool_article, n_articles, hist_article, H, lg, pos_out, val_out};
  const size_t smem = lg > 0 ? sizeof(int) << lg : 0;
  void (*kern)(const PoolTopkArgs) = n_models > 1 ? pool_topk_kernel<true> : pool_topk_kernel<false>;
  static DeviceOnce configured[2];                         // function attributes are per device
  if (configured[n_models > 1].first_time())
    NRM_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(sizeof(int) << POOL_HASH_LG_MAX)));
  kern<<<B, POOL_THREADS, smem, s>>>(args);
  NRM_LAUNCH_CHECK("pool_topk_kernel");
  return NRM_OK;
}

}  // namespace nrm

using namespace nrm;

extern "C" int nrm_pool_topk(const float* logits, int n_models, long long model_stride, int B, int N, int k, const int* pool_article,
                             int n_articles, const int* hist_article, int H, int* pos_out, float* val_out, void* stream) {
  if (!logits || !pool_article || !pos_out || !val_out) { set_error("nrm_pool_topk: null pointer"); return NRM_EINVAL; }
  if (B <= 0 || N <= 0 || n_articles <= 0) { set_error("nrm_pool_topk: B, N, n_articles must be positive (got %d, %d, %d)", B, N, n_articles); return NRM_EINVAL; }
  return launch_pool_topk(logits, n_models, model_stride, B, N, k, pool_article, n_articles, hist_article, H, pos_out, val_out,
                          (cudaStream_t)stream);
}
