// Feature-row kernels: decode the packed float64 rows, gather the embedding tables
// (reference: user_invariant_interest_model.py:58-79, user_instant_interest_model.py:20-23)
// and, for the backward, build sorted segments of table ids and reduce the row gradients
// into the tables without atomics on floating-point data.
#include "nrm_kernels.cuh"

namespace nrm {

// ---------------------------------------------------------------------------------
// embed_rows_kernel: 8 threads per row, 32 rows per CTA.
//   history row  -> xin_h[row, 0:66] = [cat+mean(sub) 32 | relu(sent) 16 | type 8 | time 8 | rt | scroll]
//   target row   -> e[row, 136:200] = same first 64 columns, e[row, 200:264] = pca (fp32),
//                   e[row, 128:136] = relu(Linear(3,8)(x_global row))
// Rows are addressed as one list: [0, NH) history, [NH, NH+R) targets.
// When keys32/keys8 are non-null the decoded table ids are also written as sort keys.
// ---------------------------------------------------------------------------------
// One row's decoded fields, from either wire format (the compact one: nrm_wire.cu; float32 article rows hold exactly the
// values `x.to(float32)` gives the reference, so both formats produce the same bits)
struct RowFields {
  int tix[4], cat, sub[5], typ;
  float s0, s1, s2;
};
// position of history row r, or of candidate row r (impression r / C, column r % C), in the compact id arrays
__device__ __forceinline__ long long compact_index(const CompactPtrs& ca, bool is_hist, long long r, int C) {
  return is_hist ? r : (long long)((int)r / C) * ca.cand_bs + (int)r % C;
}
__device__ __forceinline__ const float* compact_article(const CompactPtrs& ca, bool is_hist, long long r) {
  int art = is_hist ? ca.hist_article[r] : ca.cand_article[r];
  art = (art < 0 || art >= ca.n_articles) ? 0 : art;         // out-of-range ids read the pad article (as nrm_expand_compact does)
  return ca.articles + (long long)art * 80;
}

template <bool COMPACT>
__global__ void __launch_bounds__(256)
embed_rows_kernel(const double* __restrict__ xh, const double* __restrict__ xt, long long xt_bs,
                  const double* __restrict__ xg, long long xg_bs, const CompactPtrs ca, int H, int C, long long NH, long long N,
                  const float* __restrict__ P, float* __restrict__ xin_h, float* __restrict__ e, float* __restrict__ pca_h,
                  int* __restrict__ keys32, int* __restrict__ keys8) {
  pdl_wait();                                          // programmatic dependent launch: see nrm_common.cuh
  pdl_trigger();
  if (COMPACT && (long long)blockIdx.x * 32 >= N) {    // tail blocks: float32 labels -> float64
    const long long i = ((long long)blockIdx.x - (N + 31) / 32) * 256 + threadIdx.x;
    if (ca.label32 != nullptr && i < (N - NH)) ca.label64[i] = (double)ca.label32[i];
    return;
  }
  const long long row = (long long)blockIdx.x * 32 + (threadIdx.x >> 3);
  const int q = threadIdx.x & 7;
  if (row >= N) return;
  const bool is_hist = row < NH;
  const double* src = nullptr;
  const float* art = nullptr;
  RowFields f;
  if (COMPACT) {
    const long long r = compact_index(ca, is_hist, is_hist ? row : row - NH, C);
    art = compact_article(ca, is_hist, r);
    const unsigned t = is_hist ? ca.hist_time[r] : ca.cand_time[r];
    f.tix[0] = (int)(t & 0xfffu); f.tix[1] = (int)((t >> 12) & 0xfu); f.tix[2] = (int)((t >> 16) & 0x1fu); f.tix[3] = (int)((t >> 21) & 0x1fu);
    const float4 c0 = __ldg(reinterpret_cast<const float4*>(art + 64)), c1 = __ldg(reinterpret_cast<const float4*>(art + 68));
    const float2 c2 = __ldg(reinterpret_cast<const float2*>(art + 72));
    f.cat = (int)c0.x; f.sub[0] = (int)c0.y; f.sub[1] = (int)c0.z; f.sub[2] = (int)c0.w; f.sub[3] = (int)c1.x; f.sub[4] = (int)c1.y;
    f.s0 = c1.z; f.s1 = c1.w; f.s2 = c2.x; f.typ = (int)c2.y;
  } else {
    if (is_hist) {
      src = xh + row * HC;
    } else {
      const long long r = row - NH;
      src = xt + (r / C) * xt_bs + (r % C) * TC;
    }
    // ids are exact integers stored as doubles; float32 -> int64 truncation in the reference
#pragma unroll
    for (int i = 0; i < 4; ++i) f.tix[i] = (int)(float)src[i];
    f.cat = (int)(float)src[68];
#pragma unroll
    for (int i = 0; i < 5; ++i) f.sub[i] = (int)(float)src[69 + i];
    f.s0 = (float)src[74]; f.s1 = (float)src[75]; f.s2 = (float)src[76];
    f.typ = (int)(float)src[77];
  }
  const int cat = clampi(f.cat, 0, NCAT - 1);
  int sub[5];
#pragma unroll
  for (int i = 0; i < 5; ++i) sub[i] = clampi(f.sub[i], 0, NCAT - 1);
  const float s0 = f.s0, s1 = f.s1, s2 = f.s2;
  const int typ = clampi(f.typ, 0, NTYPE - 1);
  const int iy = clampi(f.tix[0], 0, NYEAR - 1), im = clampi(f.tix[1], 0, NMONTH - 1);
  const int id = clampi(f.tix[2], 0, NDAY - 1), ih = clampi(f.tix[3], 0, NHOUR - 1);

  // category + mean of the 5 sub-categories, columns 4q..4q+3
  const float4* tab = reinterpret_cast<const float4*>(P + P_CAT);
  const float4 c = __ldg(tab + cat * 8 + q);
  float4 s = __ldg(tab + sub[0] * 8 + q);
#pragma unroll
  for (int i = 1; i < 5; ++i) {
    const float4 v = __ldg(tab + sub[i] * 8 + q);
    s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
  }
  float4 both;
  both.x = c.x + s.x / 5.0f; both.y = c.y + s.y / 5.0f; both.z = c.z + s.z / 5.0f; both.w = c.w + s.w / 5.0f;

  // sentiment Linear(3,16)+ReLU, outputs 2q, 2q+1
  float se[2];
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const int o = 2 * q + i;
    const float* w = P + P_SENT_W + o * 3;
    float v = __ldg(P + P_SENT_B + o);
    v = fmaf(s0, __ldg(w + 0), v); v = fmaf(s1, __ldg(w + 1), v); v = fmaf(s2, __ldg(w + 2), v);
    se[i] = fmaxf(v, 0.f);
  }
  const float ty = __ldg(P + P_TYPE + typ * 8 + q);
  float tm = __ldg(P + P_YEAR + iy * 8 + q);
  tm += __ldg(P + P_MONTH + im * 8 + q);
  tm += __ldg(P + P_DAY + id * 8 + q);
  tm += __ldg(P + P_HOUR + ih * 8 + q);

  float* dst = is_hist ? (xin_h + row * XIN) : (e + (row - NH) * E + E_XT);
  // 66-float rows are only 8-byte aligned: use float2 stores for the 4-wide group
  reinterpret_cast<float2*>(dst + 4 * q)[0] = make_float2(both.x, both.y);
  reinterpret_cast<float2*>(dst + 4 * q)[1] = make_float2(both.z, both.w);
  reinterpret_cast<float2*>(dst + 32 + 2 * q)[0] = make_float2(se[0], se[1]);
  dst[48 + q] = ty;
  dst[56 + q] = tm;
  if (is_hist) {
    if (q < 2) dst[64 + q] = COMPACT ? __ldg(ca.hist_click + row * 2 + q) : (float)src[78 + q];
    if (pca_h != nullptr) {
      // text/img PCA slice as fp32 [NH, 64] (what `x_history.to(float32)` gives the reference, user_invariant_interest_model.py:74):
      // the attention kernels of both branches then stage plain fp32 rows, and the input rows are read exactly once per step
      float4* pd = reinterpret_cast<float4*>(pca_h + row * 64 + q * 8);
      if (COMPACT) {
        pd[0] = __ldg(reinterpret_cast<const float4*>(art + q * 8));
        pd[1] = __ldg(reinterpret_cast<const float4*>(art + q * 8) + 1);
      } else {
        const double2* ps = reinterpret_cast<const double2*>(src + 4 + q * 8);
        const double2 a = ps[0], b = ps[1], c2 = ps[2], d = ps[3];
        pd[0] = make_float4((float)a.x, (float)a.y, (float)b.x, (float)b.y);
        pd[1] = make_float4((float)c2.x, (float)c2.y, (float)d.x, (float)d.y);
      }
    }
  } else {
    const long long r = row - NH;
    float* er = e + r * E;
    // pca columns 4..67 -> e[200:264]; 8 threads x 8 values
    float g0, g1, g2;
    if (COMPACT) {
      reinterpret_cast<float4*>(er + E_PCAT + q * 8)[0] = __ldg(reinterpret_cast<const float4*>(art + q * 8));
      reinterpret_cast<float4*>(er + E_PCAT + q * 8)[1] = __ldg(reinterpret_cast<const float4*>(art + q * 8) + 1);
      g0 = __ldg(art + 74); g1 = __ldg(art + 75); g2 = __ldg(art + 76);
    } else {
#pragma unroll
      for (int i = 0; i < 8; ++i) er[E_PCAT + q * 8 + i] = (float)src[4 + q * 8 + i];
      const double* gsrc = xg + (r / C) * xg_bs + (r % C) * GC;
      g0 = (float)gsrc[0]; g1 = (float)gsrc[1]; g2 = (float)gsrc[2];
    }
    // instant-interest: relu(W g + b), output q
    const float* w = P + P_INST_W + q * 3;
    float v = __ldg(P + P_INST_B + q);
    v = fmaf(g0, __ldg(w + 0), v); v = fmaf(g1, __ldg(w + 1), v); v = fmaf(g2, __ldg(w + 2), v);
    er[E_INST + q] = fmaxf(v, 0.f);
  }
  if (keys32 != nullptr && q == 0) {
    int* k32 = keys32 + row * 6;
    k32[0] = cat;
#pragma unroll
    for (int i = 0; i < 5; ++i) k32[1 + i] = sub[i];
    int* k8 = keys8 + row * 5;
    k8[0] = K8_TYPE + typ; k8[1] = K8_YEAR + iy; k8[2] = K8_MONTH + im; k8[3] = K8_DAY + id; k8[4] = K8_HOUR + ih;
  }
}

// ---------------------------------------------------------------------------------
// Deterministic counting sort of table ids.  Both streams are sorted by the same launches:
//   stream 0: keys32 (6 per row: category + 5 sub-categories, keys < 3000)
//   stream 1: keys8  (5 per row: type / year / month / day / hour, keys < 185)
//   sort_hist:    per 2048-entry chunk, histogram of keys                    -> chunk_hist[chunk][key]
//   sort_colscan: per key (a warp each), exclusive scan over chunks (in place) + key totals
//   sort_keyscan: per stream (a CTA each), exclusive scan over keys of the totals -> seg[0..nkeys] (segment
//                 starts), the same for the number of SEG_GROUP-sized groups, and the group -> key map
//   sort_scatter: stable rank of each entry inside its chunk + the two offsets -> perm
// Integer atomics are used only for counts (order independent).
// ---------------------------------------------------------------------------------
struct SortStream {
  const int* keys; long long n; int nkeys; int nchunks;
  int* chunk_hist; int* seg; int* gkey; int* perm;
};
struct SortPair { SortStream s[2]; };

__global__ void __launch_bounds__(1024)
sort_hist_kernel(const SortPair sp) {
  pdl_wait();                                          // programmatic dependent launch: see nrm_common.cuh
  pdl_trigger();
  extern __shared__ int hist[];
  const int st = blockIdx.x < sp.s[0].nchunks ? 0 : 1;
  const SortStream& S = sp.s[st];
  const int chunk = blockIdx.x - (st ? sp.s[0].nchunks : 0);
  for (int i = threadIdx.x; i < S.nkeys; i += blockDim.x) hist[i] = 0;
  __syncthreads();
  const long long base = (long long)chunk * SORT_CHUNK;
  for (int i = threadIdx.x; i < SORT_CHUNK; i += blockDim.x)
    if (base + i < S.n) atomicAdd(&hist[S.keys[base + i]], 1);
  __syncthreads();
  int* out = S.chunk_hist + (long long)chunk * S.nkeys;
  for (int i = threadIdx.x; i < S.nkeys; i += blockDim.x) out[i] = hist[i];
}

// Per key (one warp each): exclusive scan of the chunk histograms over chunks, in place, and the key's total.
__global__ void __launch_bounds__(256)
sort_colscan_kernel(const SortPair sp) {
  pdl_wait();                                          // programmatic dependent launch: see nrm_common.cuh
  pdl_trigger();
  int key = blockIdx.x * 8 + (threadIdx.x >> 5);
  const int st = key < sp.s[0].nkeys ? 0 : 1;
  const SortStream& S = sp.s[st];
  if (st) key -= sp.s[0].nkeys;
  const int lane = threadIdx.x & 31;
  if (key >= S.nkeys) return;
  int* totals = S.seg + 2 * (S.nkeys + 1);
  int carry = 0;
  for (int c0 = 0; c0 < S.nchunks; c0 += 32) {
    const int c = c0 + lane;
    int* p = S.chunk_hist + (long long)c * S.nkeys + key;
    const int own = (c < S.nchunks) ? *p : 0;
    int v = own;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, v, o); if (lane >= o) v += t; }
    if (c < S.nchunks) *p = carry + v - own;
    carry += __shfl_sync(0xffffffffu, v, 31);
  }
  if (lane == 0) totals[key] = carry;
}

// One CTA per stream: exclusive scan over keys of the totals -> segment starts, and of the number of
// SEG_GROUP-sized groups -> group starts; also the group -> key map.
__global__ void __launch_bounds__(1024)
sort_keyscan_kernel(const SortPair sp) {
  pdl_wait();                                          // programmatic dependent launch: see nrm_common.cuh
  pdl_trigger();
  __shared__ int warp_off[2][32];
  __shared__ int block_tot[2];
  __shared__ int carry[2];
  const SortStream& S = sp.s[blockIdx.x];
  const int nkeys = S.nkeys;
  const int* totals = S.seg + 2 * (nkeys + 1);
  int* seg_start = S.seg;
  int* grp_start = S.seg + nkeys + 1;
  int* group_key = S.gkey;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  if (threadIdx.x == 0) { carry[0] = 0; carry[1] = 0; }
  __syncthreads();
  for (int k0 = 0; k0 < nkeys; k0 += 1024) {
    const int key = k0 + threadIdx.x;
    const int total = key < nkeys ? totals[key] : 0;
    const int vals[2] = {total, (total + SEG_GROUP - 1) / SEG_GROUP};
    int excl[2];
#pragma unroll
    for (int s = 0; s < 2; ++s) {
      int v = vals[s];
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, v, o); if (lane >= o) v += t; }
      if (lane == 31) warp_off[s][wid] = v;      // inclusive warp total
      excl[s] = v - vals[s];
    }
    __syncthreads();
    if (wid == 0) {
#pragma unroll
      for (int s = 0; s < 2; ++s) {
        const int own = warp_off[s][lane];
        int v = own;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, v, o); if (lane >= o) v += t; }
        warp_off[s][lane] = v - own;               // exclusive offset of each warp
        if (lane == 31) block_tot[s] = v;
      }
    }
    __syncthreads();
    const int off0 = carry[0] + warp_off[0][wid] + excl[0];
    const int off1 = carry[1] + warp_off[1][wid] + excl[1];
    if (key < nkeys) {
      seg_start[key] = off0;
      grp_start[key] = off1;
      for (int gi = 0; gi < vals[1]; ++gi) group_key[off1 + gi] = key;
    }
    __syncthreads();
    if (threadIdx.x == 0) { carry[0] += block_tot[0]; carry[1] += block_tot[1]; }
    __syncthreads();
  }
  if (threadIdx.x == 0) { seg_start[nkeys] = carry[0]; grp_start[nkeys] = carry[1]; }
}

// One CTA (4 warps) per chunk.  All warps first stage the chunk's keys and the per-key base position
// (segment start + offset of this chunk inside the segment) in shared memory; then warp 0 walks the entries in
// order, 32 at a time: entries with equal keys inside a round are ranked with match_any, earlier rounds through
// the shared counter.  The walk touches shared memory and registers only.
__global__ void __launch_bounds__(128)
sort_scatter_kernel(const SortPair sp) {
  pdl_wait();                                          // programmatic dependent launch: see nrm_common.cuh
  pdl_trigger();
  extern __shared__ int ssm[];                      // keys[SORT_CHUNK] | pos[nkeys] | segment starts[nkeys]
  const int st = blockIdx.x < sp.s[0].nchunks ? 0 : 1;
  const SortStream& S = sp.s[st];
  const int chunk = blockIdx.x - (st ? sp.s[0].nchunks : 0);
  int* skeys = ssm;
  int* pos = ssm + SORT_CHUNK;
  const long long base = (long long)chunk * SORT_CHUNK;
  const int total = (int)min((long long)SORT_CHUNK, S.n - base);
  const int* cb = S.chunk_hist + (long long)chunk * S.nkeys;      // exclusive per-chunk offsets
  // stage keys, segment starts and this chunk's offsets with 4-byte cp.async: every request is in flight at once
  int* segs = pos + S.nkeys;                        // scratch copy of the segment starts
  auto cp4 = [](int* dst, const int* src) {
    const unsigned d = (unsigned)__cvta_generic_to_shared(dst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"(d), "l"(src) : "memory");
  };
  for (int i = threadIdx.x; i < total; i += 128) cp4(skeys + i, S.keys + base + i);
  for (int i = threadIdx.x; i < S.nkeys; i += 128) { cp4(pos + i, cb + i); cp4(segs + i, S.seg + i); }
  asm volatile("cp.async.wait_all;\n" ::: "memory");
  __syncthreads();
  for (int i = threadIdx.x; i < S.nkeys; i += 128) pos[i] += segs[i];
  __syncthreads();
  if (threadIdx.x >= 32) return;
  const int lane = threadIdx.x;
  for (int r0 = 0; r0 < total; r0 += 32) {
    const int i = r0 + lane;
    const bool valid = i < total;
    const int key = valid ? skeys[i] : (S.nkeys + lane);           // distinct dummy keys never match
    const unsigned peers = __match_any_sync(0xffffffffu, key);
    const int leader = __ffs(peers) - 1;
    const int rank = __popc(peers & ((1u << lane) - 1u));
    int before = 0;
    if (valid && lane == leader) { before = pos[key]; pos[key] = before + __popc(peers); }
    before = __shfl_sync(0xffffffffu, before, leader);
    if (valid) S.perm[before + rank] = (int)(base + i);
    __syncwarp();
  }
}

// ---------------------------------------------------------------------------------
// Segment reduction of row gradients into table rows.
//   entry id -> (row, slot); source vector = dsrc(row)[col0 + col], weight by slot.
//   level 1: one warp per group of <= SEG_GROUP sorted entries (all of one key)
//   level 2: one warp per key sums its groups in order and writes the table gradient row
// W = 32: category table (6 entries per row: cat weight 1, five sub-categories weight 1/5)
// W = 8 : type / year / month / day / hour tables (5 entries per row)
// ---------------------------------------------------------------------------------
template <int W>
__device__ __forceinline__ float seg_load(int entry, const float* __restrict__ dxin_h, const float* __restrict__ dxt,
                                          long long NH, int col) {
  constexpr int SLOTS = (W == 32) ? 6 : 5;
  const int row = entry / SLOTS, slot = entry - row * SLOTS;
  const int c = (W == 32) ? col : ((slot == 0 ? 48 : 56) + col);
  const float v = (row < NH) ? __ldg(dxin_h + (long long)row * XIN + c) : __ldg(dxt + ((long long)row - NH) * D + c);
  return (W == 32 && slot != 0) ? v / 5.0f : v;     // d mean(sub)/d sub_i = 1/5
}

// The group's entry ids are fetched with one coalesced load per 32 entries and handed around with shuffles, so the
// row loads of a group are independent of each other (8 in flight per lane) instead of chained behind perm[i].
template <int W>
__device__ __forceinline__ void table_grad_l1(const SortStream& S, int g, const float* __restrict__ dxin_h,
                                              const float* __restrict__ dxt, long long NH, float* __restrict__ gpart) {
  const int* seg_start = S.seg;
  const int* grp_start = S.seg + S.nkeys + 1;
  const int lane = threadIdx.x & 31;
  const int key = S.gkey[g];
  const int beg = seg_start[key] + (g - grp_start[key]) * SEG_GROUP;
  const int end = min(beg + SEG_GROUP, seg_start[key + 1]);
  const int n = end - beg;
  int ids[SEG_GROUP / 32];
#pragma unroll
  for (int q = 0; q < SEG_GROUP / 32; ++q) ids[q] = (q * 32 + lane < n) ? S.perm[beg + q * 32 + lane] : 0;
  if (W == 32) {
    float acc = 0.f;
#pragma unroll
    for (int q = 0; q < SEG_GROUP / 32; ++q) {
      const int m = min(32, n - q * 32);
      if (m <= 0) break;
      int i = 0;
      for (; i + 16 <= m; i += 16) {
        float v[16];
#pragma unroll
        for (int u = 0; u < 16; ++u) v[u] = seg_load<32>(__shfl_sync(0xffffffffu, ids[q], i + u), dxin_h, dxt, NH, lane);
#pragma unroll
        for (int u = 0; u < 16; ++u) acc += v[u];
      }
      for (; i + 4 <= m; i += 4) {
        float v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) v[u] = seg_load<32>(__shfl_sync(0xffffffffu, ids[q], i + u), dxin_h, dxt, NH, lane);
#pragma unroll
        for (int u = 0; u < 4; ++u) acc += v[u];
      }
      for (; i < m; ++i) acc += seg_load<32>(__shfl_sync(0xffffffffu, ids[q], i), dxin_h, dxt, NH, lane);
    }
    gpart[(long long)g * 32 + lane] = acc;
  } else {
    // four entries per step (8 lanes each); the four interleaved partial sums are combined in a fixed order
    const int sub = lane >> 3, col = lane & 7;
    float acc = 0.f;
#pragma unroll
    for (int q = 0; q < SEG_GROUP / 32; ++q) {
      const int m = min(32, n - q * 32);
      if (m <= 0) break;
      for (int i = 0; i < m; i += 8) {
        float v[2];
#pragma unroll
        for (int u = 0; u < 2; ++u) {
          const int j = i + 4 * u + sub;
          const int id = __shfl_sync(0xffffffffu, ids[q], j & 31);
          v[u] = (j < m) ? seg_load<8>(id, dxin_h, dxt, NH, col) : 0.f;
        }
        acc += v[0]; acc += v[1];
      }
    }
    const float a1 = __shfl_down_sync(0xffffffffu, acc, 8);
    const float a2 = __shfl_down_sync(0xffffffffu, acc, 16);
    const float a3 = __shfl_down_sync(0xffffffffu, acc, 24);
    if (sub == 0) gpart[(long long)g * 8 + col] = ((acc + a1) + a2) + a3;
  }
}

// groups of stream 0 first (grid sized from upper bounds; surplus warps exit)
__global__ void __launch_bounds__(256)
table_grad_l1_kernel(const SortPair sp, int warps0, const float* __restrict__ dxin_h, const float* __restrict__ dxt,
                     long long NH, float* __restrict__ gpart32, float* __restrict__ gpart8) {
  pdl_wait();                                          // programmatic dependent launch: see nrm_common.cuh
  pdl_trigger();
  const int w = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (w < warps0) {
    const SortStream& S = sp.s[0];
    if (w < S.seg[2 * S.nkeys + 1]) table_grad_l1<32>(S, w, dxin_h, dxt, NH, gpart32);
  } else {
    const SortStream& S = sp.s[1];
    const int g = w - warps0;
    if (g < S.seg[2 * S.nkeys + 1]) table_grad_l1<8>(S, g, dxin_h, dxt, NH, gpart8);
  }
}

// Level 2.  32-wide table: one CTA (4 warps) per key -- the padding id 0 of the sub-category slots collects ~40 % of
// all entries (>1000 groups), so its groups are split in four contiguous ranges, each summed by one warp with 8
// independent loads in flight, and the four partial sums are combined in warp order.  8-wide tables: one warp per
// 4 keys (at most ~150 groups each).
__global__ void __launch_bounds__(128)
table_grad_l2_kernel(const SortPair sp, const float* __restrict__ gpart32, const float* __restrict__ gpart8,
                     float* __restrict__ grads) {
  pdl_wait();                                          // programmatic dependent launch: see nrm_common.cuh
  pdl_trigger();
  __shared__ float red[4][32];
  const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (blockIdx.x < NKEY32) {
    const int key = blockIdx.x;
    const int* grp_start = sp.s[0].seg + NKEY32 + 1;
    const int g0 = grp_start[key], g1 = grp_start[key + 1];
    const int per = (g1 - g0 + 3) / 4;
    const int a = g0 + wid * per, b = min(g1, a + per);
    float acc = 0.f;
    int g = a;
    for (; g + 8 <= b; g += 8) {
      float v[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) v[u] = gpart32[(long long)(g + u) * 32 + lane];
#pragma unroll
      for (int u = 0; u < 8; ++u) acc += v[u];
    }
    for (; g < b; ++g) acc += gpart32[(long long)g * 32 + lane];
    red[wid][lane] = acc;
    __syncthreads();
    if (wid == 0) grads[P_CAT + (long long)key * 32 + lane] = ((red[0][lane] + red[1][lane]) + red[2][lane]) + red[3][lane];
  } else {
    const int key = ((blockIdx.x - NKEY32) * 4 + wid) * 4 + (lane >> 3), col = lane & 7;
    if (key >= NKEY8) return;
    const int* grp_start = sp.s[1].seg + NKEY8 + 1;
    const int g0 = grp_start[key], g1 = grp_start[key + 1];
    float acc = 0.f;
    int g = g0;
    for (; g + 4 <= g1; g += 4) {
      const float v0 = gpart8[(long long)g * 8 + col], v1 = gpart8[(long long)(g + 1) * 8 + col];
      const float v2 = gpart8[(long long)(g + 2) * 8 + col], v3 = gpart8[(long long)(g + 3) * 8 + col];
      acc += v0; acc += v1; acc += v2; acc += v3;
    }
    for (; g < g1; ++g) acc += gpart8[(long long)g * 8 + col];
    float* dst;
    if (key < K8_YEAR) dst = grads + P_TYPE + (long long)(key - K8_TYPE) * 8;
    else if (key < K8_MONTH) dst = grads + P_YEAR + (long long)(key - K8_YEAR) * 8;
    else if (key < K8_DAY) dst = grads + P_MONTH + (long long)(key - K8_MONTH) * 8;
    else if (key < K8_HOUR) dst = grads + P_DAY + (long long)(key - K8_DAY) * 8;
    else dst = grads + P_HOUR + (long long)(key - K8_HOUR) * 8;
    dst[col] = acc;
  }
}

// ---------------------------------------------------------------------------------
// Sentiment Linear(3,16)+ReLU and instant Linear(3,8)+ReLU gradients.
// One LANE per row: it loads its row's 3 sentiment inputs, 16 activations and 16 upstream gradients (11 independent
// 16/24-byte loads), and keeps all 16 x 4 products (column 3 = bias) in registers over its rows; the 32 lanes of a warp
// are then summed with shuffles in lane order, the warps of a CTA in warp order.  Target rows add the 8 x 4 products
// of the instant-interest layer.
// part[blockIdx.x][0:64]  = sentiment (o*4 + i), part[..][64:96] = instant (o*4 + i)
// ---------------------------------------------------------------------------------
template <bool COMPACT>
__global__ void __launch_bounds__(256)
small_linear_grad_kernel(const double* __restrict__ xh, const double* __restrict__ xt, long long xt_bs,
                         const double* __restrict__ xg, long long xg_bs, const CompactPtrs ca, int C, long long NH, long long N,
                         const float* __restrict__ xin_h, const float* __restrict__ e,
                         const float* __restrict__ dxin_h, const float* __restrict__ dxt, const float* __restrict__ de,
                         float* __restrict__ part) {
  pdl_wait();                                          // programmatic dependent launch: see nrm_common.cuh
  pdl_trigger();
  __shared__ float red[8][96];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float as[16][4], ai[8][4];
#pragma unroll
  for (int o = 0; o < 16; ++o)
#pragma unroll
    for (int i = 0; i < 4; ++i) as[o][i] = 0.f;
#pragma unroll
  for (int o = 0; o < 8; ++o)
#pragma unroll
    for (int i = 0; i < 4; ++i) ai[o][i] = 0.f;
  const long long stride = (long long)gridDim.x * 256;
  for (long long row = (long long)blockIdx.x * 256 + threadIdx.x; row < N; row += stride) {
    const bool is_hist = row < NH;
    const long long r = row - NH;
    const float* actp = is_hist ? (xin_h + row * XIN + 32) : (e + r * E + E_XT + 32);
    const float* dvp = is_hist ? (dxin_h + row * XIN + 32) : (dxt + r * D + 32);
    float in[3], gl[3] = {0.f, 0.f, 0.f};
    if (COMPACT) {
      const float* art = compact_article(ca, is_hist, compact_index(ca, is_hist, is_hist ? row : r, C));
      const float2 a = __ldg(reinterpret_cast<const float2*>(art + 70));      // sentiment 70-72
      in[0] = a.x; in[1] = a.y; in[2] = __ldg(art + 72);
      if (!is_hist) { gl[0] = __ldg(art + 74); gl[1] = __ldg(art + 75); gl[2] = __ldg(art + 76); }
    } else {
      const double* src = is_hist ? (xh + row * HC) : (xt + (r / C) * xt_bs + (r % C) * TC);
      const double2 s01 = __ldg(reinterpret_cast<const double2*>(src + 74));     // columns 74, 75 (16-byte aligned: rows are 640 / 624 B)
      in[0] = (float)s01.x; in[1] = (float)s01.y; in[2] = (float)__ldg(src + 76);
      if (!is_hist) {
        const double* gsrc = xg + (r / C) * xg_bs + (r % C) * GC;
        gl[0] = (float)__ldg(gsrc); gl[1] = (float)__ldg(gsrc + 1); gl[2] = (float)__ldg(gsrc + 2);
      }
    }
    float act[16], dv[16];
    if (is_hist) {                                   // 66-float rows: 8-byte aligned
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        const float2 a = __ldg(reinterpret_cast<const float2*>(actp) + q), d = __ldg(reinterpret_cast<const float2*>(dvp) + q);
        act[2 * q] = a.x; act[2 * q + 1] = a.y; dv[2 * q] = d.x; dv[2 * q + 1] = d.y;
      }
    } else {
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const float4 a = __ldg(reinterpret_cast<const float4*>(actp) + q), d = __ldg(reinterpret_cast<const float4*>(dvp) + q);
        act[4 * q] = a.x; act[4 * q + 1] = a.y; act[4 * q + 2] = a.z; act[4 * q + 3] = a.w;
        dv[4 * q] = d.x; dv[4 * q + 1] = d.y; dv[4 * q + 2] = d.z; dv[4 * q + 3] = d.w;
      }
    }
#pragma unroll
    for (int o = 0; o < 16; ++o) {
      const float dpre = act[o] > 0.f ? dv[o] : 0.f;
      as[o][0] = fmaf(dpre, in[0], as[o][0]); as[o][1] = fmaf(dpre, in[1], as[o][1]);
      as[o][2] = fmaf(dpre, in[2], as[o][2]); as[o][3] += dpre;
    }
    if (!is_hist) {
      const float g0 = gl[0], g1 = gl[1], g2 = gl[2];
      const float4 ia0 = __ldg(reinterpret_cast<const float4*>(e + r * E + E_INST)), ia1 = __ldg(reinterpret_cast<const float4*>(e + r * E + E_INST) + 1);
      const float4 di0 = __ldg(reinterpret_cast<const float4*>(de + r * E + E_INST)), di1 = __ldg(reinterpret_cast<const float4*>(de + r * E + E_INST) + 1);
      const float iav[8] = {ia0.x, ia0.y, ia0.z, ia0.w, ia1.x, ia1.y, ia1.z, ia1.w};
      const float div[8] = {di0.x, di0.y, di0.z, di0.w, di1.x, di1.y, di1.z, di1.w};
#pragma unroll
      for (int o = 0; o < 8; ++o) {
        const float dpi = iav[o] > 0.f ? div[o] : 0.f;
        ai[o][0] = fmaf(dpi, g0, ai[o][0]); ai[o][1] = fmaf(dpi, g1, ai[o][1]);
        ai[o][2] = fmaf(dpi, g2, ai[o][2]); ai[o][3] += dpi;
      }
    }
  }
  // lanes -> warp (xor tree: fixed shape), warps -> CTA (warp order)
#pragma unroll
  for (int o = 0; o < 16; ++o)
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      float v = as[o][i];
#pragma unroll
      for (int sft = 16; sft > 0; sft >>= 1) v += __shfl_xor_sync(0xffffffffu, v, sft);
      if (lane == 0) red[warp][o * 4 + i] = v;
    }
#pragma unroll
  for (int o = 0; o < 8; ++o)
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      float v = ai[o][i];
#pragma unroll
      for (int sft = 16; sft > 0; sft >>= 1) v += __shfl_xor_sync(0xffffffffu, v, sft);
      if (lane == 0) red[warp][64 + o * 4 + i] = v;
    }
  __syncthreads();
  if (threadIdx.x < 96) {
    const int k = threadIdx.x;
    float v = red[0][k];
#pragma unroll
    for (int q = 1; q < 8; ++q) v += red[q][k];
    part[(long long)blockIdx.x * 96 + k] = v;
  }
}

// One block per output k (96): every thread sums a strided share of the per-CTA partials, then a fixed-shape tree in shared
// memory (deterministic) and the scatter of the [96] vector into the flat gradient entries.
__global__ void __launch_bounds__(256)
small_linear_grad_finish_kernel(const float* __restrict__ part, int nparts, float* __restrict__ grads) {
  pdl_wait();                                          // programmatic dependent launch: see nrm_common.cuh
  pdl_trigger();
  __shared__ float red[256];
  const int k = blockIdx.x, t = threadIdx.x;
  float acc = 0.f;
#pragma unroll 4
  for (int p = t; p < nparts; p += 256) acc += part[(long long)p * 96 + k];
  red[t] = acc;
  __syncthreads();
#pragma unroll
  for (int o = 128; o > 0; o >>= 1) {
    if (t < o) red[t] += red[t + o];
    __syncthreads();
  }
  if (t != 0) return;
  acc = red[0];
  if (k < 64) {
    const int o = k >> 2, i = k & 3;
    if (i < 3) grads[P_SENT_W + o * 3 + i] = acc; else grads[P_SENT_B + o] = acc;
  } else {
    const int o = (k - 64) >> 2, i = k & 3;
    if (i < 3) grads[P_INST_W + o * 3 + i] = acc; else grads[P_INST_B + o] = acc;
  }
}

// ---------------------------------------------------------------------------------
// host-side launchers
// ---------------------------------------------------------------------------------
int launch_embed_rows(const BatchPtrs& in, const float* P, Workspace& w, bool with_keys, cudaStream_t s) {
  const int grid = (int)((w.N + 31) / 32);
  const CompactPtrs& ca = in.compact;
  if (ca.articles != nullptr) {
    const int tail = ca.label32 != nullptr ? (int)((w.R + 255) / 256) : 0;       // label conversion blocks ([B,C] dense labels: cand_bs == C)
    launch_pdl(embed_rows_kernel<true>, dim3(grid + tail), dim3(256), 0, s, in.xh, in.xt, in.xt_bs, in.xg, in.xg_bs, ca, w.H, w.C, w.NH, w.N, P, w.xin_h, w.e, w.pca_h, with_keys ? w.keys32 : nullptr, with_keys ? w.keys8 : nullptr);
  } else {
    launch_pdl(embed_rows_kernel<false>, dim3(grid), dim3(256), 0, s, in.xh, in.xt, in.xt_bs, in.xg, in.xg_bs, ca, w.H, w.C, w.NH, w.N, P, w.xin_h, w.e, w.pca_h, with_keys ? w.keys32 : nullptr, with_keys ? w.keys8 : nullptr);
  }
  NRM_LAUNCH_CHECK("embed_rows_kernel");
  return NRM_OK;
}

static SortPair make_sort_pair(Workspace& w) {
  SortPair sp;
  const long long n32 = w.N * 6, n8 = w.N * 5;
  sp.s[0] = SortStream{w.keys32, n32, NKEY32, (int)((n32 + SORT_CHUNK - 1) / SORT_CHUNK), w.chunk_hist32, w.seg32, w.gkey32, w.perm32};
  sp.s[1] = SortStream{w.keys8, n8, NKEY8, (int)((n8 + SORT_CHUNK - 1) / SORT_CHUNK), w.chunk_hist8, w.seg8, w.gkey8, w.perm8};
  return sp;
}

// The sort only depends on the ids decoded by embed_rows_kernel; the table gradients need it at the very end.
int launch_table_sort(Workspace& w, cudaStream_t s) {
  const SortPair sp = make_sort_pair(w);
  const int nch = sp.s[0].nchunks + sp.s[1].nchunks;
  static DeviceOnce configured;                          // function attributes are per device
  if (configured.first_time()) {
    NRM_CUDA(cudaFuncSetAttribute(sort_scatter_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(sizeof(int) * (SORT_CHUNK + 2 * NKEY32))));
  }
  launch_pdl(sort_hist_kernel, dim3(nch), dim3(1024), NKEY32 * sizeof(int), s, sp);
  NRM_LAUNCH_CHECK("sort_hist_kernel");
  launch_pdl(sort_colscan_kernel, dim3((NKEY32 + NKEY8 + 7) / 8), dim3(256), 0, s, sp);
  NRM_LAUNCH_CHECK("sort_colscan_kernel");
  launch_pdl(sort_keyscan_kernel, dim3(2), dim3(1024), 0, s, sp);
  NRM_LAUNCH_CHECK("sort_keyscan_kernel");
  launch_pdl(sort_scatter_kernel, dim3(nch), dim3(128), sizeof(int) * (SORT_CHUNK + 2 * NKEY32), s, sp);
  NRM_LAUNCH_CHECK("sort_scatter_kernel");
  return NRM_OK;
}

int launch_table_grads(Workspace& w, float* grads, cudaStream_t s) {
  const SortPair sp = make_sort_pair(w);
  const long long g32 = sp.s[0].n / SEG_GROUP + NKEY32 + 1, g8 = sp.s[1].n / SEG_GROUP + NKEY8 + 1;   // upper bounds
  { KernelTimer t("table_l1", s);
  launch_pdl(table_grad_l1_kernel, dim3((int)((g32 + g8 + 7) / 8)), dim3(256), 0, s, sp, (int)g32, w.dxin_h, w.dxt, w.NH, w.gpart32, w.gpart8);
  NRM_LAUNCH_CHECK("table_grad_l1_kernel"); }
  { KernelTimer t("table_l2", s);
  launch_pdl(table_grad_l2_kernel, dim3(NKEY32 + (NKEY8 + 15) / 16), dim3(128), 0, s, sp, w.gpart32, w.gpart8, grads);
  NRM_LAUNCH_CHECK("table_grad_l2_kernel"); }
  return NRM_OK;
}

int launch_small_linear_grads(const BatchPtrs& in, Workspace& w, float* grads, cudaStream_t s) {
  // one row per lane and pass: enough CTAs to cover the rows once, at most one wave of 2 CTAs per SM
  int nparts = (int)((w.N + 255) / 256);
  nparts = max(1, min(nparts, min(1024, 2 * sm_count())));
  const CompactPtrs& ca = in.compact;
  if (ca.articles != nullptr)
    launch_pdl(small_linear_grad_kernel<true>, dim3(nparts), dim3(256), 0, s, in.xh, in.xt, in.xt_bs, in.xg, in.xg_bs, ca, w.C, w.NH, w.N, w.xin_h, w.e, w.dxin_h, w.dxt, w.de, w.small_part);
  else
    launch_pdl(small_linear_grad_kernel<false>, dim3(nparts), dim3(256), 0, s, in.xh, in.xt, in.xt_bs, in.xg, in.xg_bs, ca, w.C, w.NH, w.N, w.xin_h, w.e, w.dxin_h, w.dxt, w.de, w.small_part);
  NRM_LAUNCH_CHECK("small_linear_grad_kernel");
  launch_pdl(small_linear_grad_finish_kernel, dim3(96), dim3(256), 0, s, w.small_part, nparts, grads);
  NRM_LAUNCH_CHECK("small_linear_grad_finish_kernel");
  return NRM_OK;
}

}  // namespace nrm
