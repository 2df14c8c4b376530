// Pool negatives for training (nrm_sample_negatives): k extra candidates per impression, drawn from an article pool on the device,
// so that a captured training step draws fresh ones at every replay.  The rules are those of include/nrm_b200.h; in short, attempt a
// of impression b at step t draws pool position n = first n with cdf[n] > r, r = (u * total) >> 64, u the first 64 bits of
// Philox4x32-10(counter (a, row_offset + b, t lo, t hi), key (seed lo, seed hi)); an id already in the impression's history, its own
// candidates or its accepted negatives is rejected; attempts run in order until k acceptances or 32 k attempts.
//
// One warp per impression.  The exclusion set (history, own candidates, then every accepted negative) lives in an open-addressing
// table in shared memory with nrm_recommend.cu's hash, at load factor <= 1/2.  The 32 lanes evaluate 32 consecutive attempts at
// once: a lane's draw is a candidate if it passes the table; __match_any_sync keeps only the lowest lane of each repeated id and a
// ballot numbers the survivors in attempt order, so the accepted ids and their columns are those of the sequential rule.  A round
// that accepts more than the remaining k drops its later survivors, as the sequential rule stops there.
#include "nrm_kernels.cuh"

namespace nrm {

constexpr int NEG_K_MAX = 64;
constexpr int NEG_SET_MAX = 16384;            // H + C0 + k: the exclusion table's entries (nrm_recommend.cu's history limit)
constexpr int NEG_HASH_LG_MAX = 15;           // 32768 slots, 128 KB
constexpr int NEG_WARPS = 4;                  // impressions per CTA, fewer when their tables would need more than 128 KB
constexpr int NEG_ATTEMPTS_PER_K = 32;

struct NegArgs {
  const int* hist_article; int H;
  int* cand_article; unsigned* cand_time; float* label32;
  int B, C, C0, k;
  const int* pool_article; const long long* cdf; int N, n_articles;
  unsigned long long seed; const long long* step; int row_offset;
  int hash_lg, warps;
};

// Philox4x32-10 (Salmon et al., SC'11; the Random123 constants)
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 key) {
#pragma unroll
  for (int i = 0; i < 10; ++i) {
    const unsigned lo0 = 0xD2511F53u * c.x, hi0 = __umulhi(0xD2511F53u, c.x);
    const unsigned lo1 = 0xCD9E8D57u * c.z, hi1 = __umulhi(0xCD9E8D57u, c.z);
    c = make_uint4(hi1 ^ c.y ^ key.x, lo1, hi0 ^ c.w ^ key.y, lo0);
    key.x += 0x9E3779B9u; key.y += 0xBB67AE85u;
  }
  return c;
}

__device__ __forceinline__ bool neg_contains(const int* tab, int lg, int id) {
  const unsigned m = (1u << lg) - 1;
  for (unsigned h = pool_hash(id, lg);; h = (h + 1) & m) {
    const int v = tab[h];
    if (v == id) return true;
    if (v == 0) return false;
  }
}

// ids outside [1, n_articles) are never drawn, so they need no entry
__device__ __forceinline__ void neg_insert(int* tab, int lg, int id, int n_articles) {
  if (id < 1 || id >= n_articles) return;
  const unsigned m = (1u << lg) - 1;
  for (unsigned h = pool_hash(id, lg);; h = (h + 1) & m) {
    const int old = atomicCAS(&tab[h], 0, id);
    if (old == 0 || old == id) return;
  }
}

__global__ void __launch_bounds__(NEG_WARPS * 32)
sample_negatives_kernel(const NegArgs a) {
  pdl_wait();
  pdl_trigger();
  extern __shared__ int neg_tab[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.x * a.warps + warp;
  if (b >= a.B) return;
  const unsigned below = (1u << lane) - 1;
  int* art = a.cand_article + (long long)b * a.C;
  unsigned* tim = a.cand_time + (long long)b * a.C;
  float* lab = a.label32 + (long long)b * a.C;
  int first = -1;                                            // the impression's first positive column
  for (int c0 = 0; c0 < a.C0 && first < 0; c0 += 32) {
    const unsigned m = __ballot_sync(0xffffffffu, c0 + lane < a.C0 && lab[c0 + lane] > 0.f);
    if (m) first = c0 + __ffs(m) - 1;
  }
  const long long total = a.cdf[a.N - 1];
  int acc = 0;
  if (first >= 0 && total > 0) {
    const unsigned t_pos = tim[first];
    const int lg = a.hash_lg;
    int* tab = neg_tab + (warp << lg);
    for (int i = lane; i < (1 << lg); i += 32) tab[i] = 0;
    __syncwarp();
    for (int h = lane; h < a.H; h += 32) neg_insert(tab, lg, a.hist_article[(long long)b * a.H + h], a.n_articles);
    for (int c = lane; c < a.C0; c += 32) neg_insert(tab, lg, art[c], a.n_articles);
    __syncwarp();
    const unsigned long long t = (unsigned long long)*a.step;
    const uint2 key = make_uint2((unsigned)a.seed, (unsigned)(a.seed >> 32));
    const unsigned row = (unsigned)(a.row_offset + b);
    for (int base = 0; base < NEG_ATTEMPTS_PER_K * a.k && acc < a.k; base += 32) {
      const uint4 x = philox4x32_10(make_uint4((unsigned)(base + lane), row, (unsigned)t, (unsigned)(t >> 32)), key);
      const unsigned long long r = __umul64hi((unsigned long long)x.x | ((unsigned long long)x.y << 32), (unsigned long long)total);
      int lo = 0, hi = a.N - 1;                              // first n with cdf[n] > r (cdf[N - 1] = total > r)
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if ((unsigned long long)__ldg(a.cdf + mid) > r) hi = mid; else lo = mid + 1;
      }
      const int id = __ldg(a.pool_article + lo);
      const bool ok = id >= 1 && id < a.n_articles && !neg_contains(tab, lg, id);
      const unsigned same = __match_any_sync(0xffffffffu, ok ? id : -1 - lane);
      const bool take = ok && (same & below) == 0;            // the first attempt of this round to draw the id
      const unsigned taken = __ballot_sync(0xffffffffu, take);
      const int slot = acc + __popc(taken & below);
      if (take && slot < a.k) {
        art[a.C0 + slot] = id;
        tim[a.C0 + slot] = t_pos;
        lab[a.C0 + slot] = 0.f;
        neg_insert(tab, lg, id, a.n_articles);
      }
      acc = min(a.k, acc + __popc(taken));
      __syncwarp();
    }
  }
  for (int s = acc + lane; s < a.k; s += 32) {               // what was not accepted: pad columns
    art[a.C0 + s] = 0;
    tim[a.C0 + s] = 0u;
    lab[a.C0 + s] = 0.f;
  }
}

int launch_sample_negatives(const NegArgs& args, cudaStream_t s) {
  NegArgs a = args;
  const int entries = a.H + a.C0 + a.k;
  a.hash_lg = 5;
  while ((1 << a.hash_lg) < 2 * entries) ++a.hash_lg;
  a.warps = NEG_WARPS;
  while (a.warps > 1 && (a.warps << a.hash_lg) > (1 << NEG_HASH_LG_MAX)) a.warps >>= 1;
  const size_t smem = sizeof(int) * ((size_t)a.warps << a.hash_lg);
  static DeviceOnce configured;                            // function attributes are per device
  if (configured.first_time())
    NRM_CUDA(cudaFuncSetAttribute(sample_negatives_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)(sizeof(int) << NEG_HASH_LG_MAX)));
  NRM_CUDA(launch_pdl(sample_negatives_kernel, dim3((unsigned)((a.B + a.warps - 1) / a.warps)), dim3(a.warps * 32), smem, s, a));
  NRM_LAUNCH_CHECK("sample_negatives_kernel");
  return NRM_OK;
}

}  // namespace nrm

using namespace nrm;

extern "C" int nrm_sample_negatives(const int* hist_article, int H, int* cand_article, unsigned* cand_time, float* label32, int B, int C,
                                    int C0, const int* pool_article, const long long* pool_cdf, int N, int n_articles,
                                    unsigned long long seed, const long long* step, int row_offset, void* stream) {
  if (!hist_article || !cand_article || !cand_time || !label32 || !pool_article || !pool_cdf || !step) {
    set_error("nrm_sample_negatives: null pointer");
    return NRM_EINVAL;
  }
  if (B <= 0 || H <= 0 || C0 <= 0 || N <= 0 || n_articles <= 0) {
    set_error("nrm_sample_negatives: B, H, C0, N, n_articles must be positive (got %d, %d, %d, %d, %d)", B, H, C0, N, n_articles);
    return NRM_EINVAL;
  }
  const int k = C - C0;
  if (C <= C0 || k > NEG_K_MAX) { set_error("nrm_sample_negatives: need 1 <= C - C0 <= %d (got C = %d, C0 = %d)", NEG_K_MAX, C, C0); return NRM_EINVAL; }
  if ((long long)H + C > NEG_SET_MAX) { set_error("nrm_sample_negatives: need H + C <= %d (got H = %d, C = %d)", NEG_SET_MAX, H, C); return NRM_EINVAL; }
  if (row_offset < 0 || (long long)row_offset + B > 0x7fffffffLL) {
    set_error("nrm_sample_negatives: need 0 <= row_offset and row_offset + B < 2^31 (got %d, %d)", row_offset, B);
    return NRM_EINVAL;
  }
  const NegArgs a{hist_article, H, cand_article, cand_time, label32, B, C, C0, k, pool_article, pool_cdf, N, n_articles, seed, step, row_offset,
                  0, 0};
  return launch_sample_negatives(a, (cudaStream_t)stream);
}
