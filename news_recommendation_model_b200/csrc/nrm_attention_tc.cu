// The tensor-core attention's work outside the row-stacked kernels (nrm_attention_rs.cu, nrm_attention_rs_bwd.cu), for precision
// bf16 / bf16x3, plus the tcgen05 building-block test and micro-benchmark.  Reduced algebra: DESIGN.md section 3.
//   candidate_tp_kernel          tp = Bm t + b1 per candidate row, before the forward
//   attention_finish_kernel      sums the row-stacked backward's per-CTA partials into dA, dWd, dw2, db2, and runs the tp path of
//                                the backward (dBm, db1 partials; dxt += dtp Bm) over the candidate rows
//   attention_tp_finish_kernel   sums the tp-path partials into dBm, dBm - dA and db1
//   umma_selftest_kernel         nrm_debug_umma_selftest (tests/test_gpu_tensorcore.py)
//   mma_microbench_kernel        nrm_debug_mma_microbench (tools/mma_microbench.py)
#include "nrm_kernels.cuh"

#include "nrm_umma.cuh"

namespace nrm {

constexpr int TC_THREADS = 256;       // 8 warps: warp w reads TMEM sub-partition w & 3 and accumulator columns 32 (w >> 2) .. +32

// tp[branch][r][j] = b1[j] + sum_k (Wb + Wc)[j][k] t[r][k] for every candidate row r (t = the candidate's label
// features / PCA vector inside e_concat).  32 rows per CTA, blockIdx.y = branch.
__global__ void __launch_bounds__(256)
candidate_tp_kernel(const float* __restrict__ P, const float* __restrict__ e, long long R, float* __restrict__ tp_all) {
  pdl_wait();                                          // programmatic dependent launch: see nrm_common.cuh
  pdl_trigger();
  __shared__ float st[32][65];          // t rows
  __shared__ float sBT[64][65];         // Bm^T: [k][j]
  const AttOffsets off = blockIdx.y == 0 ? ATT_LABEL : ATT_TI;
  const int toff = blockIdx.y == 0 ? E_XT : E_PCAT;
  const float* W = P + off.fc1_w;
  float* tp = tp_all + (long long)blockIdx.y * R * 64;
  const int tid = threadIdx.x;
  const long long r0 = (long long)blockIdx.x * 32;
  const int nr = (int)min(32LL, R - r0);
  for (int i = tid; i < 32 * 64; i += 256) {
    const int r = i >> 6, k = i & 63;
    st[r][k] = r < nr ? __ldg(e + (r0 + r) * E + toff + k) : 0.f;
  }
  for (int i = tid; i < 64 * 64; i += 256) {
    const int j = i >> 6, k = i & 63;
    sBT[k][j] = __ldg(W + j * 256 + 64 + k) + __ldg(W + j * 256 + 128 + k);
  }
  __syncthreads();
  const int r = tid >> 3, jq = tid & 7;          // thread owns j = jq + 8 i
  float v[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) v[i] = __ldg(P + off.fc1_b + jq + 8 * i);
#pragma unroll 4
  for (int k = 0; k < 64; ++k) {
    const float tv = st[r][k];
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = fmaf(sBT[k][jq + 8 * i], tv, v[i]);
  }
  if (r < nr) {
#pragma unroll
    for (int i = 0; i < 8; ++i) tp[(r0 + r) * 64 + jq + 8 * i] = v[i];
  }
}

// per-CTA partial sums of the row-stacked backward (floats, ATT_TC_PARTIAL per CTA): dA^T [64 k][64 j] | dWd^T [64][64] | dw2 [64] | db2 [1]
constexpr int TCP_DA = 0, TCP_DWD = 4096, TCP_DW2 = 2 * 4096, TCP_DB2 = 2 * 4096 + 64;

// Sum the per-CTA partials (fixed order) and write the attention-MLP gradients that do not depend on tp:
//   fc1.weight grad blocks: [:, 0:64] = dA, [:, 192:256] = dWd   (the Bm-dependent blocks are completed by
//   the tp-path blocks of attention_finish_kernel + attention_tp_finish_kernel); fc2.weight = dw2; fc2.bias = db2.   Partials are transposed ([k][j]).
constexpr int COMPOSE_BLOCKS = 65;      // 64 blocks of 64 (k,j) entries + one for fc2
__device__ __forceinline__ void
attention_tc_compose_block(int block, const float* __restrict__ part_all, int nparts0, int nparts1, float* __restrict__ grads,
                           float* __restrict__ dA_all) {
  const int branch = blockIdx.y;
  const AttOffsets off = branch == 0 ? ATT_LABEL : ATT_TI;
  const float* part = part_all + (long long)branch * ATT_TC_PARTS_MAX * ATT_TC_PARTIAL;
  const int nparts = branch == 0 ? nparts0 : nparts1;
  float* dA_out = dA_all + branch * 4096;
  // block = 64 consecutive (k,j) entries (two per lane) x 32 interleaved groups of partials, combined in group order;
  // 64 such blocks (+1) per branch, so that the whole finish kernel is one wave
  __shared__ float red[32][4][32];
  const int lane = threadIdx.x & 31, grp = threadIdx.x >> 5;
  if (block < COMPOSE_BLOCKS - 1) {
    const int i = block * 64 + lane;              // k*64 + j; the lane's second entry is i + 32
    float dA0 = 0.f, dWd0 = 0.f, dA1 = 0.f, dWd1 = 0.f;
#pragma unroll 4
    for (int p = grp; p < nparts; p += 32) {
      const float* q = part + (long long)p * ATT_TC_PARTIAL;
      dA0 += q[TCP_DA + i]; dA1 += q[TCP_DA + i + 32];
      dWd0 += q[TCP_DWD + i]; dWd1 += q[TCP_DWD + i + 32];
    }
    red[grp][0][lane] = dA0; red[grp][1][lane] = dWd0; red[grp][2][lane] = dA1; red[grp][3][lane] = dWd1;
    __syncthreads();
    if (grp < 2) {                                     // warp 0 finishes entry i, warp 1 entry i + 32
      float dA = red[0][2 * grp][lane], dWd = red[0][2 * grp + 1][lane];
#pragma unroll
      for (int g = 1; g < 32; ++g) { dA += red[g][2 * grp][lane]; dWd += red[g][2 * grp + 1][lane]; }
      const int ii = i + 32 * grp;
      const int k = ii >> 6, j = ii & 63;
      float* rowp = grads + off.fc1_w + j * 256;
      rowp[k] = dA; rowp[192 + k] = dWd;
      dA_out[j * 64 + k] = dA;
    }
  } else {
    // fc2.weight (64 sums) and fc2.bias: 65 entries x 8 groups of partials
    const int ent = threadIdx.x & 127, g8 = threadIdx.x >> 7;
    float* r2 = &red[0][0][0];                         // [8][128]
    float w = 0.f;
    if (ent <= 64) {
#pragma unroll 4
      for (int p = g8; p < nparts; p += 8) w += part[(long long)p * ATT_TC_PARTIAL + (ent < 64 ? TCP_DW2 + ent : TCP_DB2)];
    }
    r2[g8 * 128 + ent] = w;
    __syncthreads();
    if (g8 == 0 && ent <= 64) {
      w = r2[ent];
#pragma unroll
      for (int g = 1; g < 8; ++g) w += r2[g * 128 + ent];
      if (ent < 64) grads[off.fc2_w + ent] = w; else grads[off.fc2_b] = w;
    }
  }
}

// The tp = Bm t + b1 path, over the R candidate rows: dBm[j][k] = sum_r dtp[r][j] t[r][k], db1[j] = sum_r dtp[r][j],
// and (label branch) dxt[r][k] += sum_j dtp[r][j] Bm[j][k].  32 rows per CTA -> partials, summed by the finish kernel.
constexpr int TPG_ROWS = 32, TPG_PART = 4096 + 64, TPG_SUB = 4;
struct TpgSmem {
  float sB[64][65];                   // Bm[j][k] = Wb + Wc (shared by the block's four tiles)
  float sd[TPG_SUB][TPG_ROWS][65];    // dtp rows
  float st[TPG_SUB][TPG_ROWS][64];    // t rows
};
// 1024 threads = four groups of 256, each taking one 32-row tile (partial number block * 4 + group)
__device__ __forceinline__ void
attention_tp_grad_block(int block, TpgSmem& sm, const float* __restrict__ dtp_all, const float* __restrict__ e, long long R,
                        const float* __restrict__ P, float* __restrict__ dxt, float* __restrict__ part_all, int nparts) {
  const int branch = blockIdx.y;
  const float* dtp = dtp_all + (long long)branch * R * 64;
  const int toff = branch == 0 ? E_XT : E_PCAT;
  const float* W = P + (branch == 0 ? ATT_LABEL.fc1_w : ATT_TI.fc1_w);     // fc1.weight [64,256]
  const int input_grads = branch == 0;
  const int nblocks = (nparts + TPG_SUB - 1) / TPG_SUB;                    // one partial per BLOCK: its four tiles are added in tile order
  float* part = part_all + (long long)branch * nblocks * TPG_PART;
  const int sub = threadIdx.x >> 8, tid = threadIdx.x & 255;
  const int tile = block * TPG_SUB + sub;
  float (*sd)[65] = sm.sd[sub];
  float (*st)[64] = sm.st[sub];
  const long long r0 = (long long)tile * TPG_ROWS;
  const int nr = (int)max(0LL, min((long long)TPG_ROWS, R - r0));          // 0 for a tile past the end: it contributes zeros
  for (int i = tid; i < TPG_ROWS * 64; i += 256) {
    const int r = i >> 6, k = i & 63;
    sd[r][k] = r < nr ? __ldg(dtp + (r0 + r) * 64 + k) : 0.f;
    st[r][k] = r < nr ? __ldg(e + (r0 + r) * E + toff + k) : 0.f;
  }
  if (input_grads)
    for (int i = threadIdx.x; i < 64 * 64; i += 1024) {
      const int j = i >> 6, k = i & 63;
      sm.sB[j][k] = __ldg(W + j * 256 + 64 + k) + __ldg(W + j * 256 + 128 + k);
    }
  __syncthreads();
  // dBm partial: thread (tj, tk) owns a 4 x 4 block of [j][k]
  const int tj = tid >> 4, tk = tid & 15;
  float acc[4][4];
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b) acc[a][b] = 0.f;
  float b1[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 4
  for (int r = 0; r < TPG_ROWS; ++r) {
    const float dv[4] = {sd[r][4 * tj], sd[r][4 * tj + 1], sd[r][4 * tj + 2], sd[r][4 * tj + 3]};
    const float4 tk4 = *reinterpret_cast<const float4*>(&st[r][4 * tk]);
    const float tv[4] = {tk4.x, tk4.y, tk4.z, tk4.w};
#pragma unroll
    for (int a = 0; a < 4; ++a) {
      b1[a] += dv[a];
#pragma unroll
      for (int b = 0; b < 4; ++b) acc[a][b] = fmaf(dv[a], tv[b], acc[a][b]);
    }
  }
  if (input_grads) {
    // dxt[r][k] += sum_j dtp[r][j] Bm[j][k]; thread (r, kq) owns k = kq + 8 i
    const int r = tid >> 3, kq = tid & 7;
    float v[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll 4
    for (int j = 0; j < 64; ++j) {
      const float d = sd[r][j];
#pragma unroll
      for (int i = 0; i < 8; ++i) v[i] = fmaf(d, sm.sB[j][kq + 8 * i], v[i]);
    }
    if (r < nr) {
#pragma unroll
      for (int i = 0; i < 8; ++i) dxt[(r0 + r) * 64 + kq + 8 * i] += v[i];
    }
  }
  // the four tiles of the block: tiles 1-3 hand their sums over through shared memory (the row buffers are free now), tile 0 adds
  // them in tile order and writes the block's partial
  __syncthreads();
  float* xch = &sm.sd[0][0][0];                                             // >= 3 * TPG_PART floats (sd and st are contiguous)
  static_assert(sizeof(TpgSmem::sd) + sizeof(TpgSmem::st) >= 3 * TPG_PART * sizeof(float), "exchange area");
  if (sub > 0) {
    float* o = xch + (sub - 1) * TPG_PART;
#pragma unroll
    for (int a = 0; a < 4; ++a) {
      *reinterpret_cast<float4*>(o + (4 * tj + a) * 64 + 4 * tk) = make_float4(acc[a][0], acc[a][1], acc[a][2], acc[a][3]);
      if (tk == 0) o[4096 + 4 * tj + a] = b1[a];
    }
  }
  __syncthreads();
  if (sub == 0) {
    float* out = part + (long long)block * TPG_PART;
#pragma unroll
    for (int a = 0; a < 4; ++a) {
      float4 v = make_float4(acc[a][0], acc[a][1], acc[a][2], acc[a][3]);
      float bb = b1[a];
#pragma unroll
      for (int t = 0; t < 3; ++t) {
        const float4 x = *reinterpret_cast<const float4*>(xch + t * TPG_PART + (4 * tj + a) * 64 + 4 * tk);
        v.x += x.x; v.y += x.y; v.z += x.z; v.w += x.w;
        bb += xch[t * TPG_PART + 4096 + 4 * tj + a];
      }
      *reinterpret_cast<float4*>(out + (4 * tj + a) * 64 + 4 * tk) = v;
      if (tk == 0) out[4096 + 4 * tj + a] = bb;
    }
  }
}

// One launch for the two independent reductions: the first ceil(nparts / 4) blocks take 4 x 32 candidate rows each through
// the tp path (they are the longer ones, so they are scheduled first), the next 65 sum the per-CTA partials of the
// backward kernels.

__global__ void __launch_bounds__(1024)
attention_finish_kernel(const float* __restrict__ part_all, int nparts0, int nparts1, float* __restrict__ grads, float* __restrict__ dA_all,
                        const float* __restrict__ dtp_all, const float* __restrict__ e, long long R, const float* __restrict__ P,
                        float* __restrict__ dxt, float* __restrict__ tp_part, int nparts) {
  pdl_wait();                                          // programmatic dependent launch: see nrm_common.cuh
  pdl_trigger();
  extern __shared__ __align__(16) unsigned char fin_raw[];
  const int tp_blocks = (nparts + TPG_SUB - 1) / TPG_SUB;
  if ((int)blockIdx.x < tp_blocks) {
    attention_tp_grad_block(blockIdx.x, *reinterpret_cast<TpgSmem*>(fin_raw), dtp_all, e, R, P, dxt, tp_part, nparts);
  } else {
    attention_tc_compose_block(blockIdx.x - tp_blocks, part_all, nparts0, nparts1, grads, dA_all);
  }
}

// fc1.weight grad blocks [:, 64:128] = dBm and [:, 128:192] = dBm - dA; fc1.bias = db1.
// block = 64 consecutive entries x 4 interleaved groups of partials, combined in group order
__global__ void __launch_bounds__(256)
attention_tp_finish_kernel(const float* __restrict__ part_all, int nparts, const float* __restrict__ dA_all,
                           float* __restrict__ grads) {
  pdl_wait();                                          // programmatic dependent launch: see nrm_common.cuh
  pdl_trigger();
  const int branch = blockIdx.y;
  const AttOffsets off = branch == 0 ? ATT_LABEL : ATT_TI;
  const float* part = part_all + (long long)branch * nparts * TPG_PART;
  const float* dA = dA_all + branch * 4096;
  __shared__ float red[4][64];
  const int lane = threadIdx.x & 63, grp = threadIdx.x >> 6;
  const int i = blockIdx.x * 64 + lane;              // 0 .. 4096+64, grid = 65 blocks
  float s = 0.f;
  for (int p = grp; p < nparts; p += 4) s += part[(long long)p * TPG_PART + i];
  red[grp][lane] = s;
  __syncthreads();
  if (grp != 0) return;
  s = ((red[0][lane] + red[1][lane]) + red[2][lane]) + red[3][lane];
  if (i < 4096) {
    const int j = i >> 6, k = i & 63;
    grads[off.fc1_w + j * 256 + 64 + k] = s;
    grads[off.fc1_w + j * 256 + 128 + k] = s - dA[i];
  } else {
    grads[off.fc1_b + (i - 4096)] = s;
  }
}

template <int NP> struct TileBytes { static constexpr uint32_t T64 = NP * umma::TILE64_BYTES; };   // one [64][64] operand tile, all parts

// ---------------------------------------------------------------------------------
// Self test of the tensor-core building blocks (tests/test_gpu_tensorcore.py): four 64x64x64 products with the
// interleaved half-lane accumulators:
//   out[0] = a0 b0^T (K-major x K-major)      out[1] = a1 b1^T (upper half-lanes)
//   out[2] = a0^T b0 (both tiles read MN-major)   out[3] = a1 b1^T... see below
// mode 0: K-major / K-major;  mode 1: A MN-major, B MN-major (out = a^T b);  mode 2: A K-major, B MN-major (out = a b)
// split = 1 or 3.
// ---------------------------------------------------------------------------------
template <int SPLIT>
__global__ void __launch_bounds__(TC_THREADS)
umma_selftest_kernel(const float* __restrict__ a0, const float* __restrict__ a1, const float* __restrict__ b0,
                     const float* __restrict__ b1, float* __restrict__ out, int mode) {
  constexpr int NP = SPLIT == 3 ? 2 : 1;
  extern __shared__ __align__(128) unsigned char st_raw[];
  unsigned char* opA[2] = {st_raw, st_raw + TileBytes<NP>::T64};
  unsigned char* opB[2] = {st_raw + 2 * TileBytes<NP>::T64, st_raw + 3 * TileBytes<NP>::T64};
  uint64_t* mbar = reinterpret_cast<uint64_t*>(st_raw + 4 * TileBytes<NP>::T64);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(mbar + 1);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const float* srcs[4] = {a0, a1, b0, b1};
  for (int m = 0; m < 4; ++m) {
    unsigned char* tile = m < 2 ? opA[m] : opB[m - 2];
    for (int it = tid; it < 64 * 8; it += TC_THREADS) {
      const int r = it & 63, kb = it >> 6;
      float v[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) v[i] = srcs[m][r * 64 + kb * 8 + i];
      umma::store_operand8<NP>(tile, umma::tile64_offset(r, kb), umma::TILE64_BYTES, v);
    }
  }
  if (warp == 0) umma::tmem_alloc(tmem_slot, 64);
  if (tid == 0) umma::mbar_init(mbar, 1);
  umma::fence_async_smem();
  umma::fence_before_sync();
  __syncthreads();
  umma::fence_after_sync();
  const uint32_t tmem = *tmem_slot;
  if (warp == 0 && umma::elect_one()) {
    for (int q = 0; q < 2; ++q) {
      const uint32_t d = tmem + ((uint32_t)(16 * q) << 16);
      const uint32_t aa = umma::smem_u32(opA[q]), bb = umma::smem_u32(opB[q]);
      if (mode == 0) umma::mma_product<SPLIT, 4>(d, umma::op_tile64_k(aa), umma::op_tile64_k(bb), umma::make_idesc_bf16(64, 64), false);
      else if (mode == 1) umma::mma_product<SPLIT, 4>(d, umma::op_tile64_mn(aa), umma::op_tile64_mn(bb), umma::make_idesc_bf16(64, 64, true, true), false);
      else umma::mma_product<SPLIT, 4>(d, umma::op_tile64_k(aa), umma::op_tile64_mn(bb), umma::make_idesc_bf16(64, 64, false, true), false);
    }
    umma::mma_commit(mbar);
  }
  umma::mbar_wait(mbar, 0);
  umma::fence_after_sync();
  // warp w reads sub-partition w & 3, column half w >> 2
  const int half = lane >> 4, row = (warp & 3) * 16 + (lane & 15), cb = warp >> 2;
  {
    float v[32];
    umma::tmem_ld32(tmem + ((uint32_t)((warp & 3) * 32) << 16) + cb * 32, v);
#pragma unroll
    for (int j = 0; j < 32; ++j) out[(half * 64 + row) * 64 + cb * 32 + j] = v[j];
  }
  umma::fence_before_sync();
  __syncthreads();
  if (warp == 0) umma::tmem_dealloc(tmem, 64);
}

// ---------------------------------------------------------------------------------
// launchers
// ---------------------------------------------------------------------------------
// needs the candidate rows of e written by embed_rows_kernel
int launch_candidate_tp(const float* P, Workspace& w, cudaStream_t s) {
  launch_pdl(candidate_tp_kernel, dim3(dim3((unsigned)((w.R + 31) / 32), 2)), dim3(256), 0, s, P, w.e, w.R, w.tp);
  NRM_LAUNCH_CHECK("candidate_tp_kernel");
  return NRM_OK;
}

// both branches at once (after both backward kernels)
int launch_attention_finish_tc(const float* P, Workspace& w, float* grads, cudaStream_t s) {
  const int nparts = (int)((w.R + TPG_ROWS - 1) / TPG_ROWS);
  static DeviceOnce configured;                          // function attributes are per device
  if (configured.first_time()) {
    NRM_CUDA(cudaFuncSetAttribute(attention_finish_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(TpgSmem)));
  }
  launch_pdl(attention_finish_kernel, dim3(COMPOSE_BLOCKS + (nparts + TPG_SUB - 1) / TPG_SUB, 2), dim3(1024), sizeof(TpgSmem), s, w.att_part, w.att_tc_parts[0], w.att_tc_parts[1], grads, w.att_dA, w.dtp, w.e, w.R, P, w.dxt, w.tp_part, nparts);
  NRM_LAUNCH_CHECK("attention_finish_kernel");
  launch_pdl(attention_tp_finish_kernel, dim3(dim3(TPG_PART / 64, 2)), dim3(256), 0, s, w.tp_part, (nparts + TPG_SUB - 1) / TPG_SUB, w.att_dA, grads);
  NRM_LAUNCH_CHECK("attention_tp_finish_kernel");
  return NRM_OK;
}

}  // namespace nrm

using namespace nrm;

// a0, a1, b0, b1: [64,64] fp32 (device); out: [2,64,64] fp32.  mode 0: out_q = a_q b_q^T; 1: a_q^T b_q; 2: a_q b_q.
// split 1: operands rounded to bf16; 3: hi/lo split (fp32-grade).
extern "C" int nrm_debug_umma_selftest(const float* a0, const float* a1, const float* b0, const float* b1, float* out,
                                       int mode, int split, void* stream) {
  if (!a0 || !a1 || !b0 || !b1 || !out || mode < 0 || mode > 2 || (split != 1 && split != 3)) {
    set_error("nrm_debug_umma_selftest: bad argument"); return NRM_EINVAL;
  }
  if (split == 1) {
    const size_t smem = 4 * TileBytes<1>::T64 + 64;
    NRM_CUDA(cudaFuncSetAttribute(umma_selftest_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    umma_selftest_kernel<1><<<1, TC_THREADS, smem, (cudaStream_t)stream>>>(a0, a1, b0, b1, out, mode);
  } else {
    const size_t smem = 4 * TileBytes<2>::T64 + 64;
    NRM_CUDA(cudaFuncSetAttribute(umma_selftest_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    umma_selftest_kernel<3><<<1, TC_THREADS, smem, (cudaStream_t)stream>>>(a0, a1, b0, b1, out, mode);
  }
  NRM_LAUNCH_CHECK("umma_selftest_kernel");
  return NRM_OK;
}

// ---------------------------------------------------------------------------------
// Micro-benchmark of the tensor-core building blocks (tools/mma_microbench.py): cycles (clock64 on the issuing
// thread, from first issue to mbarrier completion) for `reps` back-to-back products of `nk` K=16 steps each.
//   variant 0: M=64  N=64  K-major x K-major      1: M=64 N=64 MN x MN      2: M=128 N=64 K x K
//   variant 3: M=64  N=8   K x K                  4: only tcgen05.ld 32x32b.x32 x reps (all four warps)
// ---------------------------------------------------------------------------------
namespace nrm {
__global__ void __launch_bounds__(TC_THREADS)
mma_microbench_kernel(long long* __restrict__ out, int variant, int reps, int nk) {
  extern __shared__ __align__(128) unsigned char mb_raw[];
  unsigned char* opA = mb_raw;                       // 128 x 64 bf16 = 16 KB
  unsigned char* opB = mb_raw + 16384;               // 64 x 64 bf16 = 8 KB
  __shared__ uint64_t mbar, mbar2;
  __shared__ uint32_t tmem_slot;
  const int tid = threadIdx.x, warp = tid >> 5;
  for (int i = tid; i < (16384 + 8192) / 4; i += TC_THREADS) reinterpret_cast<uint32_t*>(mb_raw)[i] = 0x3c003c00u;
  if (warp == 0) umma::tmem_alloc(&tmem_slot, 128);
  if (tid == 0) { umma::mbar_init(&mbar, 1); umma::mbar_init(&mbar2, 1); }
  umma::fence_async_smem();
  umma::fence_before_sync();
  __syncthreads();
  umma::fence_after_sync();
  const uint32_t tmem = tmem_slot;
  long long t0 = 0, t1 = 0, t2 = 0;
  if (variant < 4) {
    if (warp == 0 && umma::elect_one()) {
      const uint32_t aa = umma::smem_u32(opA), bb = umma::smem_u32(opB);
      const uint64_t a_k = umma::make_desc(aa, 1024, 128), b_k = umma::make_desc(bb, 1024, 128);
      const uint64_t a_mn = umma::make_desc(aa, 128, 1024), b_mn = umma::make_desc(bb, 128, 1024);
      const uint64_t a_128 = umma::make_desc(aa, 2048, 128), b_8 = umma::make_desc(bb, 128, 128);
      t0 = clock64();
      for (int r = 0; r < reps; ++r) {
        if (variant == 0) {
#pragma unroll 4
          for (int ks = 0; ks < nk; ++ks) umma::mma_bf16(tmem, a_k + (uint64_t)((ks & 3) * 128), b_k + (uint64_t)((ks & 3) * 128), umma::make_idesc_bf16(64, 64), ks > 0);
        } else if (variant == 1) {
#pragma unroll 4
          for (int ks = 0; ks < nk; ++ks) umma::mma_bf16(tmem, a_mn + (uint64_t)((ks & 3) * 16), b_mn + (uint64_t)((ks & 3) * 16), umma::make_idesc_bf16(64, 64, true, true), ks > 0);
        } else if (variant == 2) {
#pragma unroll 4
          for (int ks = 0; ks < nk; ++ks) umma::mma_bf16(tmem, a_128 + (uint64_t)((ks & 3) * 256), b_k + (uint64_t)((ks & 3) * 128), umma::make_idesc_bf16(128, 64), ks > 0);
        } else {
#pragma unroll 4
          for (int ks = 0; ks < nk; ++ks) umma::mma_bf16(tmem, a_k + (uint64_t)((ks & 3) * 128), b_8 + (uint64_t)((ks & 3) * 16), umma::make_idesc_bf16(64, 8), ks > 0);
        }
      }
      t1 = clock64();
      umma::mma_commit(&mbar);
      umma::mbar_wait(&mbar, 0);
      t2 = clock64();
      out[0] = t1 - t0; out[1] = t2 - t0;
    }
    umma::mbar_wait(&mbar, 0);
  } else if (variant == 5) {
    // two issuing threads (warps 0 and 4), M64 N64 K-major each, disjoint accumulator columns
    if ((warp == 0 || warp == 4) && umma::elect_one()) {
      const uint32_t aa = umma::smem_u32(opA), bb = umma::smem_u32(opB);
      const uint64_t a_k = umma::make_desc(aa, 1024, 128), b_k = umma::make_desc(bb, 1024, 128);
      uint64_t* bar = warp == 0 ? &mbar : &mbar2;
      const uint32_t acc = tmem + (warp == 0 ? 0u : 64u);
      t0 = clock64();
      for (int r = 0; r < reps; ++r) {
#pragma unroll 4
        for (int ks = 0; ks < nk; ++ks) umma::mma_bf16(acc, a_k + (uint64_t)((ks & 3) * 128), b_k + (uint64_t)((ks & 3) * 128), umma::make_idesc_bf16(64, 64), ks > 0);
      }
      t1 = clock64();
      umma::mma_commit(bar);
      umma::mbar_wait(bar, 0);
      t2 = clock64();
      out[warp == 0 ? 0 : 2] = t1 - t0; out[warp == 0 ? 1 : 3] = t2 - t0;
    }
    umma::mbar_wait(&mbar, 0);
    umma::mbar_wait(&mbar2, 0);
  } else {
    umma::fence_after_sync();
    float acc = 0.f;
    t0 = clock64();
    for (int r = 0; r < reps; ++r) {
      float v[32];
      umma::tmem_ld32(tmem + ((uint32_t)((warp & 3) * 32) << 16) + (r & 1) * 32, v);
#pragma unroll
      for (int j = 0; j < 32; ++j) acc += v[j];
    }
    t1 = clock64();
    if (tid == 0) { out[0] = t1 - t0; out[1] = t1 - t0; }
    if (acc == 123.456f) out[2] = 1;
  }
  umma::fence_before_sync();
  __syncthreads();
  if (warp == 0) umma::tmem_dealloc(tmem, 128);
}
}  // namespace nrm

extern "C" int nrm_debug_mma_microbench(long long* out, int variant, int reps, int nk, void* stream) {
  if (!out || variant < 0 || variant > 5 || reps < 1 || nk < 1) { set_error("nrm_debug_mma_microbench: bad argument"); return NRM_EINVAL; }
  const size_t smem = 16384 + 8192;
  mma_microbench_kernel<<<1, TC_THREADS, smem, (cudaStream_t)stream>>>(out, variant, reps, nk);
  NRM_LAUNCH_CHECK("mma_microbench_kernel");
  return NRM_OK;
}
