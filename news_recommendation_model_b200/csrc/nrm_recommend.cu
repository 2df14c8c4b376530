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

// The phases both kernels share take their argument struct (PoolTopkArgs or PoolRankArgs) as a template parameter: they read only
// the pool and exclusion fields the two have in common, and each kernel keeps its own parameter layout.

// a pool id that may be recommended: in range and not clicked by this user
template <class Args>
__device__ __forceinline__ bool pool_id_ok(const Args& a, const int* tab, int id) {
  return id >= 1 && id < a.n_articles && !pool_clicked(tab, a.hash_lg, id);
}

// keys of positions n0 + j * POOL_THREADS from the logits alone (0: past the pool or a NaN logit in some model) and their ids;
// whether the id is eligible is left to the caller, which checks it only for the keys it wants
template <bool ENSEMBLE, class Args>
__device__ __forceinline__ void pool_raw_keys(const Args& a, const float* row, const float* mx, const float* sum, int n0,
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
template <bool MAX, class Args>
__device__ __forceinline__ float pool_model_partial(const Args& a, const float* row, const int* tab, int m, float vmax) {
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

// user b's clicked ids into the hash table tab[1 << hash_lg] (pad rows and ids no pool position can carry are left out); ends with
// a barrier
template <class Args>
__device__ __forceinline__ void pool_build_clicked(const Args& a, int b, int tid, int* tab) {
  if (a.hash_lg > 0) {
    const int cap = 1 << a.hash_lg;
    for (int i = tid; i < cap; i += POOL_THREADS) tab[i] = 0;
    __syncthreads();
    for (int h = tid; h < a.H; h += POOL_THREADS) {
      const int id = a.hist_article[(long long)b * a.H + h];
      if (id < 1 || id >= a.n_articles) continue;
      for (unsigned s = pool_hash(id, a.hash_lg);; s = (s + 1) & (unsigned)(cap - 1)) {
        const int old = atomicCAS(&tab[s], 0, id);
        if (old == 0 || old == id) break;
      }
    }
  }
  __syncthreads();
}

// ensemble: per model m, mx[m] / sum[m] = max and sum of exp(x - max) over the eligible positions; ends with a barrier
template <class Args>
__device__ __forceinline__ void pool_ensemble_stats(const Args& a, const float* row, const int* tab, float* mx, float* sum, float* red) {
  for (int m = 0; m < a.n_models; ++m) {
    const float vmax = pool_block_reduce<true>(pool_model_partial<true>(a, row, tab, m, 0.f), red);
    const float vsum = pool_block_reduce<false>(pool_model_partial<false>(a, row, tab, m, vmax), red);
    if (threadIdx.x == 0) { mx[m] = vmax; sum[m] = vsum; }
  }
  __syncthreads();
}

// sel[0, cnt) -> descending, bitonic over the next power of two (padded with 0 keys, which sort last); ends with a barrier
__device__ __forceinline__ void pool_sort_desc(unsigned long long* sel, int cnt, int tid) {
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

  pool_build_clicked(a, b, tid, clicked_tab);
  if (ENSEMBLE) pool_ensemble_stats(a, row, clicked_tab, mx, sum, red);

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
  pool_sort_desc(sel, cnt, tid);
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

// ---- nrm_pool_rank: where each of a user's held-out targets lands in that user's ranking of the whole pool --------------------
// The ranking is the one nrm_pool_topk returns a prefix of (same eligibility, scores and keys).  A target is rankable if its id is
// in [1, n_articles), is held by an eligible pool position, and does not repeat an id of an earlier slot of the user's target row.
// Two passes over the pool after the ensemble statistics: the first finds each target's key (ids -> first slot through a second
// hash table); the T rankable keys are then sorted, and in the second pass every eligible position finds by binary search the gap
// between consecutive target keys (and target scores) it falls into and counts itself there with a shared-memory integer atomic.
// A prefix sum over the gaps gives every target's counts, exactly and independently of timing, in O(N log P) work per user.
constexpr int POOL_TARGETS_MAX = 1024;
constexpr int TARGET_HASH_LG = 11;            // 2048 slots for <= 1024 ids: load factor <= 1/2

struct PoolRankArgs {
  const float* logits; int n_models; long long model_stride;
  int N;
  const int* pool_article; int n_articles;
  const int* hist_article; int H; int hash_lg;   // hash_lg 0: no exclusion
  const int* targets; int P;
  int* pos_out; int* rank_out; int* greater_out; int* equal_out; float* score_out; int* n_eligible_out;
};

// the first slot of the user's target row that holds `id`, -1 if none
__device__ __forceinline__ int pool_target_slot(const int* tgt_id, const int* tgt_slot, int id) {
  if (id < 1) return -1;                                   // 0 marks an empty table slot
  constexpr unsigned m = (1u << TARGET_HASH_LG) - 1;
  for (unsigned h = pool_hash(id, TARGET_HASH_LG);; h = (h + 1) & m) {
    const int v = tgt_id[h];
    if (v == id) return tgt_slot[h];
    if (v == 0) return -1;
  }
}

// lo + the number of entries of the descending run s[lo, hi) for which above(entry) holds (it holds on a prefix of the run)
template <class Above>
__device__ __forceinline__ int pool_count_above(const unsigned long long* s, int lo, int hi, Above above) {
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (above(s[mid])) lo = mid + 1; else hi = mid;
  }
  return lo;
}

// inclusive prefix sum of v[0, n) by one warp
__device__ __forceinline__ void pool_warp_scan(int* v, int n) {
  const int lane = threadIdx.x & 31;
  int carry = 0;
  for (int i0 = 0; i0 < n; i0 += 32) {
    int x = i0 + lane < n ? v[i0 + lane] : 0;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int y = __shfl_up_sync(0xffffffffu, x, o);
      if (lane >= o) x += y;
    }
    if (i0 + lane < n) v[i0 + lane] = x + carry;
    carry += __shfl_sync(0xffffffffu, x, 31);
  }
}

template <bool ENSEMBLE>
__global__ void __launch_bounds__(POOL_THREADS, 3)
pool_rank_kernel(const PoolRankArgs a) {
  extern __shared__ int clicked_tab[];                     // [1 << hash_lg] article ids, 0 = empty slot
  __shared__ int tgt_id[1 << TARGET_HASH_LG], tgt_slot[1 << TARGET_HASH_LG];   // target id -> its first slot in the row
  __shared__ unsigned long long slot_key[POOL_TARGETS_MAX];                    // per slot: the key of its position, 0 = not rankable
  __shared__ unsigned long long tkey[POOL_TARGETS_MAX];                        // the T rankable keys, descending
  // per gap j (between sorted targets j - 1 and j): eligible positions with a larger key than target j but not than j - 1, and the
  // same for score > and score >=; after the prefix sums, entry j is target j's count
  __shared__ int gap_rank[POOL_TARGETS_MAX], gap_greater[POOL_TARGETS_MAX], gap_ge[POOL_TARGETS_MAX];
  __shared__ float red[POOL_THREADS / 32 + 1];
  __shared__ float mx[POOL_MODELS_MAX], sum[POOL_MODELS_MAX];
  __shared__ unsigned s_count, s_eligible;
  const int tid = threadIdx.x, b = blockIdx.x, N = a.N, P = a.P;
  const float* row = a.logits + (long long)b * N;
  const int* trow = a.targets + (long long)b * P;

  for (int i = tid; i < (1 << TARGET_HASH_LG); i += POOL_THREADS) { tgt_id[i] = 0; tgt_slot[i] = 0x7fffffff; }
  for (int i = tid; i < POOL_TARGETS_MAX; i += POOL_THREADS) { slot_key[i] = 0ull; gap_rank[i] = 0; gap_greater[i] = 0; gap_ge[i] = 0; }
  if (tid == 0) { s_count = 0; s_eligible = 0; }
  pool_build_clicked(a, b, tid, clicked_tab);              // (its barriers also publish the initialisation above)
  for (int p = tid; p < P; p += POOL_THREADS) {
    const int id = trow[p];
    if (id < 1 || id >= a.n_articles) continue;            // pad slot or an id no pool position can rank
    for (unsigned h = pool_hash(id, TARGET_HASH_LG);; h = (h + 1) & ((1u << TARGET_HASH_LG) - 1)) {
      const int old = atomicCAS(&tgt_id[h], 0, id);
      if (old == 0 || old == id) { atomicMin(&tgt_slot[h], p); break; }
    }
  }
  if (ENSEMBLE) pool_ensemble_stats(a, row, clicked_tab, mx, sum, red);
  __syncthreads();

  // locate: every target's key (a repeated pool id: the occurrence ranked first)
#pragma unroll 1
  for (int n0 = tid; n0 < N; n0 += POOL_BATCH * POOL_THREADS) {
    unsigned long long key[POOL_BATCH];
    int id[POOL_BATCH];
    pool_raw_keys<ENSEMBLE>(a, row, mx, sum, n0, key, id);
#pragma unroll
    for (int j = 0; j < POOL_BATCH; ++j) {
      if (key[j] == 0ull) continue;
      const int slot = pool_target_slot(tgt_id, tgt_slot, id[j]);
      if (slot >= 0 && pool_id_ok(a, clicked_tab, id[j])) atomicMax(&slot_key[slot], key[j]);
    }
  }
  __syncthreads();
  for (int p = tid; p < P; p += POOL_THREADS)
    if (slot_key[p] != 0ull) tkey[atomicAdd(&s_count, 1u)] = slot_key[p];
  __syncthreads();
  const int T = (int)s_count;
  pool_sort_desc(tkey, T, tid);

  // count: the gap of every eligible position among the target keys, and among the target scores (the keys' upper 32 bits)
  unsigned n_eligible = 0;
#pragma unroll 1
  for (int n0 = tid; n0 < N; n0 += POOL_BATCH * POOL_THREADS) {
    unsigned long long key[POOL_BATCH];
    int id[POOL_BATCH];
    pool_raw_keys<ENSEMBLE>(a, row, mx, sum, n0, key, id);
#pragma unroll
    for (int j = 0; j < POOL_BATCH; ++j) {
      if (key[j] == 0ull || !pool_id_ok(a, clicked_tab, id[j])) continue;
      ++n_eligible;
      const unsigned long long k = key[j];
      const unsigned u = (unsigned)(k >> 32);
      const int gt = pool_count_above(tkey, 0, T, [u](unsigned long long t) { return (unsigned)(t >> 32) > u; });
      const int ge = pool_count_above(tkey, gt, T, [u](unsigned long long t) { return (unsigned)(t >> 32) >= u; });
      const int kge = pool_count_above(tkey, gt, ge, [k](unsigned long long t) { return t >= k; });
      if (kge < T) atomicAdd(&gap_rank[kge], 1);           // above targets kge.. (by key)
      if (ge < T) atomicAdd(&gap_greater[ge], 1);          // a larger score than targets ge..
      if (gt < T) atomicAdd(&gap_ge[gt], 1);               // a score at least that of targets gt..
    }
  }
  atomicAdd(&s_eligible, n_eligible);
  __syncthreads();
  const int warp = tid >> 5;
  if (warp == 0) pool_warp_scan(gap_rank, T);
  else if (warp == 1) pool_warp_scan(gap_greater, T);
  else if (warp == 2) pool_warp_scan(gap_ge, T);
  __syncthreads();

  for (int p = tid; p < P; p += POOL_THREADS) {
    const long long o = (long long)b * P + p;
    const unsigned long long k = slot_key[p];
    if (k != 0ull) {
      const int i = pool_count_above(tkey, 0, T, [k](unsigned long long t) { return t > k; });   // its place among the sorted keys
      a.pos_out[o] = (int)~(unsigned)k;
      a.rank_out[o] = gap_rank[i];
      a.greater_out[o] = gap_greater[i];
      a.equal_out[o] = gap_ge[i] - gap_greater[i] - 1;       // minus the target itself
      a.score_out[o] = pool_key_score(k);
    } else {
      a.pos_out[o] = -1;
      a.rank_out[o] = -1;
      a.greater_out[o] = -1;
      a.equal_out[o] = -1;
      a.score_out[o] = CUDART_NAN_F;
    }
  }
  if (tid == 0) a.n_eligible_out[b] = (int)s_eligible;
}

// the checks both entry points share; *lg: the exclusion table's log2 size (0: no exclusion)
static int pool_check_models_and_history(const char* fn, int n_models, long long model_stride, int B, int N, const int* hist_article,
                                         int H, int* lg) {
  if (n_models < 1 || n_models > POOL_MODELS_MAX) { set_error("%s: need 1 <= n_models <= %d (got %d)", fn, POOL_MODELS_MAX, n_models); return NRM_EINVAL; }
  if (n_models > 1 && model_stride < (long long)B * N) { set_error("%s: model_stride smaller than B * N", fn); return NRM_EINVAL; }
  *lg = 0;
  if (hist_article != nullptr) {
    if (H <= 0) { set_error("%s: H must be positive with hist_article (got %d)", fn, H); return NRM_EINVAL; }
    int l = 5;
    while (l <= POOL_HASH_LG_MAX && (1LL << l) < 2LL * H) ++l;
    if (l > POOL_HASH_LG_MAX) { set_error("%s: H = %d exceeds the %d history rows the exclusion table holds", fn, H, 1 << (POOL_HASH_LG_MAX - 1)); return NRM_EINVAL; }
    *lg = l;
  }
  return NRM_OK;
}

int launch_pool_topk(const float* logits, int n_models, long long model_stride, int B, int N, int k, const int* pool_article, int n_articles,
                     const int* hist_article, int H, int* pos_out, float* val_out, cudaStream_t s) {
  if (k < 1 || k > N || k > POOL_TOPK_MAX) { set_error("nrm_pool_topk: need 1 <= k <= min(N, %d) (got k = %d, N = %d)", POOL_TOPK_MAX, k, N); return NRM_EINVAL; }
  int lg;
  if (const int rc = pool_check_models_and_history("nrm_pool_topk", n_models, model_stride, B, N, hist_article, H, &lg)) return rc;
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

int launch_pool_rank(const float* logits, int n_models, long long model_stride, int B, int N, const int* pool_article, int n_articles,
                     const int* hist_article, int H, const int* targets, int P, int* pos_out, int* rank_out, int* greater_out,
                     int* equal_out, float* score_out, int* n_eligible_out, cudaStream_t s) {
  if (P < 1 || P > POOL_TARGETS_MAX) { set_error("nrm_pool_rank: need 1 <= P <= %d (got %d)", POOL_TARGETS_MAX, P); return NRM_EINVAL; }
  int lg;
  if (const int rc = pool_check_models_and_history("nrm_pool_rank", n_models, model_stride, B, N, hist_article, H, &lg)) return rc;
  const PoolRankArgs args{logits, n_models, model_stride, N, pool_article, n_articles, hist_article, H, lg, targets, P,
                          pos_out, rank_out, greater_out, equal_out, score_out, n_eligible_out};
  const size_t smem = lg > 0 ? sizeof(int) << lg : 0;
  void (*kern)(const PoolRankArgs) = n_models > 1 ? pool_rank_kernel<true> : pool_rank_kernel<false>;
  static DeviceOnce configured[2];
  if (configured[n_models > 1].first_time())
    NRM_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(sizeof(int) << POOL_HASH_LG_MAX)));
  kern<<<B, POOL_THREADS, smem, s>>>(args);
  NRM_LAUNCH_CHECK("pool_rank_kernel");
  return NRM_OK;
}

// ---- nrm_pool_diversify: greedy maximal-marginal-relevance re-ranking of a user's nrm_pool_topk candidates ----------------------
// One CTA per user, thread i owns candidate i (n_cand <= POOL_THREADS; the CTA is n_cand rounded up to a warp).  A thread keeps its
// candidate's unit PCA vector (article row columns 0-63), relevance, category (column 64), running max similarity to the picks and
// its state in registers.  Per step the winner of the last step publishes its vector and category to shared memory, every live
// candidate updates its max similarity with one 64-term dot product and its category's pick count by comparing categories, and a
// block arg-max over the keys pool_key(gain, i) picks the next candidate (unique keys: largest gain, ties to the lower index).
// Every reduction reads the warp results in one fixed order, so the picks do not depend on timing.
constexpr int PCA_COLS = 64, ARTICLE_COLS = 80, CATEGORY_COL = 64;

struct PoolDiversifyArgs {
  const int* cand_pos; const float* cand_score; int n_cand, k;
  float lambda; int max_per_category;
  const int* pool_article; int N;
  const float* article_rows; int n_articles;
  int* pos_out; float* val_out; float* gain_out;
};

// the largest v over the CTA, for every thread.  red[16] must not be read by another reduction before the barrier inside the next
// call on the same buffer: alternate two buffers between consecutive calls.
__device__ __forceinline__ unsigned long long diversify_block_max(unsigned long long v, unsigned long long* red) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const unsigned long long w = __shfl_xor_sync(0xffffffffu, v, o);
    v = w > v ? w : v;
  }
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  v = red[0];
  for (int w = 1; w < (int)(blockDim.x >> 5); ++w) v = red[w] > v ? red[w] : v;
  return v;
}

// a float's bits in an unsigned order that follows the float order (-0.0 == +0.0), as in pool_key
__device__ __forceinline__ unsigned diversify_ordered(float x) {
  const unsigned u = __float_as_uint(x + 0.0f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

__global__ void __launch_bounds__(POOL_THREADS, 1)
pool_diversify_kernel(const PoolDiversifyArgs a) {
  __shared__ unsigned long long red[2][POOL_THREADS / 32];
  __shared__ float4 pick_vec[PCA_COLS / 4];
  __shared__ int pick_cat;
  const int i = threadIdx.x, b = blockIdx.x;
  const long long o = (long long)b * a.n_cand + i;

  // this thread's candidate: a slot past n_cand, at position -1 (or one select never writes) is none
  int pos = i < a.n_cand ? a.cand_pos[o] : -1;
  const int id = pos >= 0 && pos < a.N ? __ldg(a.pool_article + pos) : 0;
  if (id < 1 || id >= a.n_articles) pos = -1;
  const float score = pos >= 0 ? a.cand_score[o] : 0.f;
  float u[PCA_COLS];
  int cat = 0;
  if (pos >= 0) {
    const float* r = a.article_rows + (long long)id * ARTICLE_COLS;
#pragma unroll
    for (int j = 0; j < PCA_COLS; ++j) u[j] = __ldg(r + j);
    cat = (int)__ldg(r + CATEGORY_COL);
  } else {
#pragma unroll
    for (int j = 0; j < PCA_COLS; ++j) u[j] = 0.f;
  }
  float ss = 0.f;
#pragma unroll
  for (int j = 0; j < PCA_COLS; ++j) ss = fmaf(u[j], u[j], ss);
  if (ss > 0.f) {                                          // an all-zero vector stays zero: similarity 0 to everything
    const float nrm = __fsqrt_rn(ss);
#pragma unroll
    for (int j = 0; j < PCA_COLS; ++j) u[j] = __fdiv_rn(u[j], nrm);
  }

  // relevance: min-max over the finite candidate scores (0 in the ordered bits: none); +inf -> 1, -inf -> 0, all equal -> 1
  const bool fin = pos >= 0 && isfinite(score);
  const unsigned long long hi = diversify_block_max(fin ? diversify_ordered(score) : 0u, red[0]);
  const unsigned long long lo = diversify_block_max(fin ? ~diversify_ordered(score) : 0u, red[1]);
  const float s_max = pool_key_score(hi << 32), s_min = pool_key_score((~lo & 0xffffffffull) << 32);
  float rel = 1.f;
  if (score == -CUDART_INF_F) rel = 0.f;
  else if (score != CUDART_INF_F && hi != 0ull && s_max > s_min) {
    const float d = __fsub_rn(s_max, s_min);
    rel = isfinite(d) ? __fdiv_rn(__fsub_rn(score, s_min), d)   // |s_max - s_min| beyond FLT_MAX: halve both operands first
                      : __fdiv_rn(__fsub_rn(0.5f * score, 0.5f * s_min), __fsub_rn(0.5f * s_max, 0.5f * s_min));
  }

  const int q = a.max_per_category;
  const float lam = a.lambda, mu = 1.f - a.lambda;
  bool live = pos >= 0;                                    // a candidate, not picked, its category below the cap
  float m = 0.f;
  int same = 0, t = 0;                                     // t: picks so far
  while (true) {
    const float gain = __fsub_rn(__fmul_rn(lam, rel), __fmul_rn(mu, m));
    const unsigned long long best = diversify_block_max(live ? pool_key(gain, i) : 0ull, red[t & 1]);
    if (best == 0ull) break;                               // nothing left that may be picked
    if (i == (int)~(unsigned)best) {
      live = false;
      const long long out = (long long)b * a.k + t;
      a.pos_out[out] = pos;
      a.val_out[out] = score;
      a.gain_out[out] = gain;
#pragma unroll
      for (int j = 0; j < PCA_COLS / 4; ++j) pick_vec[j] = make_float4(u[4 * j], u[4 * j + 1], u[4 * j + 2], u[4 * j + 3]);
      pick_cat = cat;
    }
    if (++t == a.k) break;
    __syncthreads();                                       // the pick is published; red[(t - 1) & 1] has been read by every thread
    if (live) {
      float d = 0.f;
#pragma unroll
      for (int j = 0; j < PCA_COLS / 4; ++j) {
        const float4 p = pick_vec[j];
        d = fmaf(u[4 * j], p.x, d);
        d = fmaf(u[4 * j + 1], p.y, d);
        d = fmaf(u[4 * j + 2], p.z, d);
        d = fmaf(u[4 * j + 3], p.w, d);
      }
      m = t == 1 ? d : fmaxf(m, d);                          // 0 only while nothing is picked: m may be negative
      if (q > 0 && pick_cat == cat && ++same >= q) live = false;
    }
  }
  for (int j = t + i; j < a.k; j += blockDim.x) {
    const long long out = (long long)b * a.k + j;
    a.pos_out[out] = -1;
    a.val_out[out] = CUDART_NAN_F;
    a.gain_out[out] = CUDART_NAN_F;
  }
}

int launch_pool_diversify(const int* cand_pos, const float* cand_score, int B, int n_cand, int k, float lambda, int max_per_category,
                          const int* pool_article, int N, const float* article_rows, int n_articles, int* pos_out, float* val_out,
                          float* gain_out, cudaStream_t s) {
  if (n_cand < 1 || n_cand > N || n_cand > POOL_THREADS) {
    set_error("nrm_pool_diversify: need 1 <= n_cand <= min(N, %d) (got n_cand = %d, N = %d)", POOL_THREADS, n_cand, N);
    return NRM_EINVAL;
  }
  if (k < 1 || k > n_cand) { set_error("nrm_pool_diversify: need 1 <= k <= n_cand (got k = %d, n_cand = %d)", k, n_cand); return NRM_EINVAL; }
  if (!(lambda >= 0.f && lambda <= 1.f)) { set_error("nrm_pool_diversify: need 0 <= lambda <= 1 (got %g)", (double)lambda); return NRM_EINVAL; }
  if (max_per_category < 0) { set_error("nrm_pool_diversify: max_per_category must be >= 0 (got %d)", max_per_category); return NRM_EINVAL; }
  const PoolDiversifyArgs args{cand_pos, cand_score, n_cand, k, lambda, max_per_category, pool_article, N, article_rows, n_articles,
                               pos_out, val_out, gain_out};
  pool_diversify_kernel<<<B, (n_cand + 31) / 32 * 32, 0, s>>>(args);
  NRM_LAUNCH_CHECK("pool_diversify_kernel");
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

extern "C" int nrm_pool_rank(const float* logits, int n_models, long long model_stride, int B, int N, const int* pool_article,
                             int n_articles, const int* hist_article, int H, const int* targets, int P, int* pos_out, int* rank_out,
                             int* greater_out, int* equal_out, float* score_out, int* n_eligible_out, void* stream) {
  if (!logits || !pool_article || !targets || !pos_out || !rank_out || !greater_out || !equal_out || !score_out || !n_eligible_out) {
    set_error("nrm_pool_rank: null pointer");
    return NRM_EINVAL;
  }
  if (B <= 0 || N <= 0 || n_articles <= 0) { set_error("nrm_pool_rank: B, N, n_articles must be positive (got %d, %d, %d)", B, N, n_articles); return NRM_EINVAL; }
  return launch_pool_rank(logits, n_models, model_stride, B, N, pool_article, n_articles, hist_article, H, targets, P, pos_out, rank_out,
                          greater_out, equal_out, score_out, n_eligible_out, (cudaStream_t)stream);
}

extern "C" int nrm_pool_diversify(const int* cand_pos, const float* cand_score, int B, int n_cand, int k, float lambda,
                                  int max_per_category, const int* pool_article, int N, const float* article_rows, int n_articles,
                                  int* pos_out, float* val_out, float* gain_out, void* stream) {
  if (!cand_pos || !cand_score || !pool_article || !article_rows || !pos_out || !val_out || !gain_out) {
    set_error("nrm_pool_diversify: null pointer");
    return NRM_EINVAL;
  }
  if (B <= 0 || N <= 0 || n_articles <= 0) { set_error("nrm_pool_diversify: B, N, n_articles must be positive (got %d, %d, %d)", B, N, n_articles); return NRM_EINVAL; }
  return launch_pool_diversify(cand_pos, cand_score, B, n_cand, k, lambda, max_per_category, pool_article, N, article_rows, n_articles,
                               pos_out, val_out, gain_out, (cudaStream_t)stream);
}
