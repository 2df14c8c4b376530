// Pairwise MLP attention + sum pooling, "row-stacked" tensor-core formulation (forward).
// Reference: PointwiseAttentionExpanded.forward (models/attention_model.py:52-97) and the pooling at
// models/user_invariant_interest_model.py:83-87.
//
// With fc1.weight = [Wa | Wb | Wc | Wd] over [h, t, t - h, t (.) h] (attention_model.py:81-86):
//     hid[(c,h)][j] = sum_k (t_c[k] h[k]) Wd[j][k] + sum_k h[k] A[j][k] + tp_c[j],   A = Wa - Wc,  tp_c = (Wb + Wc) t_c + b1
//     s[c][h] = w2 . gelu(hid[(c,h)][:]) + b2,          pooled[c][k] = sum_h s[c][h] h[h][k]
// i.e. ONE weight matrix W = [Wd | A] (64 x 128) is shared by every (candidate, history row) pair, and the pair only enters
// through its operand row [t_c (.) h | h] (K = 128).  So the rows (c, h) of an impression are STACKED into M = 128 tiles:
//
//   * full-rate M = 128 tcgen05.mma tiles with a CONSTANT B operand (the weights sit in shared memory for the life of the CTA;
//     nothing is rebuilt per candidate), no padding of H = 50 to 64 rows per candidate (250 of 256 rows carry work instead of
//     250 of 320: 22 % fewer GELUs);
//   * the A operand never touches shared memory: producer threads build their row in registers and write it to TENSOR MEMORY
//     (tcgen05.st), the MMA reads A from TMEM (".ts" form) and only the 2 KB weight slices from shared memory -- with the
//     hi/lo split (3 MMAs per product) an A operand in shared memory would cost more shared-memory bandwidth than the GELU
//     epilogue leaves;
//   * warp-specialised, mbarrier-only pipeline (no CTA-wide barrier inside the loop): 1 loader warp (global -> shared staging of a
//     history chunk, candidate vectors), 4 producer warps (operand rows -> TMEM, double-buffered), 1 MMA warp (one elected
//     thread issues, commits to mbarriers), 8 epilogue warps (TMEM -> registers, + tp, GELU, fc2 dot, scores), accumulators
//     double-buffered in TMEM so MMA(i + 1) runs under epilogue(i).
//
// Work unit = (branch, impression, group of <= 8 candidates); a unit walks its history in chunks of <= 64 rows; a chunk's rows
// (c, h) are stacked candidate-major into tiles of 128.  The pooled vector of a unit is a second, small product
// pooled^T[k][c] = sum_h H[h][k] s[c][h] per chunk (M = 64, N = 16, accumulated over the chunks in TMEM), as in nrm_attention_tc.cu.
//
// SPLIT = 1: bf16 operands.  SPLIT = 3: hi + lo bf16 parts, A_hi W_hi + A_hi W_lo + A_lo W_hi (fp32-grade, "bf16x3").

#include "nrm_attention_rs.cuh"

namespace nrm {
namespace rs {

#ifndef NRM_RS_SCORES_TU
__global__ void __launch_bounds__(256)
att_prep_rs_kernel(const float* __restrict__ P, unsigned char* __restrict__ img_all) {
  pdl_wait();
  pdl_trigger();
  const AttOffsets off = blockIdx.y == 0 ? ATT_LABEL : ATT_TI;
  unsigned char* img = img_all + (size_t)blockIdx.y * IMG_BRANCH_BYTES;
  const float* W = P + off.fc1_w;
  for (int i = blockIdx.x * 256 + threadIdx.x; i < 64 * 128; i += gridDim.x * 256) {
    const int j = i >> 7, kk = i & 127;
    const float v = kk < 64 ? W[j * 256 + 192 + kk] : W[j * 256 + (kk - 64)] - W[j * 256 + 128 + (kk - 64)];
    const __nv_bfloat16 h = __float2bfloat16_rn(v);
    const __nv_bfloat16 l = __float2bfloat16_rn(v - __bfloat162float(h));
    const uint32_t o = (uint32_t)(kk >> 3) * 1024u + (uint32_t)(j >> 3) * 128u + (uint32_t)(j & 7) * 16u + (uint32_t)(kk & 7) * 2u;
    *reinterpret_cast<__nv_bfloat16*>(img + o) = h;
    *reinterpret_cast<__nv_bfloat16*>(img + W_TILE + o) = l;
  }
  if (blockIdx.x == 0 && threadIdx.x < 64) {
    float* tail = reinterpret_cast<float*>(img + 2 * W_TILE);
    tail[threadIdx.x] = P[off.fc2_w + threadIdx.x];
    if (threadIdx.x == 0) tail[64] = P[off.fc2_b];
  }
}
#endif


struct Stage {
  float hf[HCH * HF_STRIDE];                       // fp32 history rows of the chunk (producers)
  __align__(128) unsigned char hbf[2][8192];       // the same rows as a K-major bf16 tile [64 h][64 k], hi | lo: operand A of the pooling product
                                                   // (read MN-major), published by the producer threads of the chunk's first candidate
  __align__(16) float tv[CG][64];                  // candidate vectors t_c
  __align__(16) float tpv[CG][64];                 // tp_c = (Wb + Wc) t_c + b1
  __align__(128) unsigned char s2[2][4096];        // scores [32 slots = candidate + 8 * column quarter][64 h] K-major bf16, hi | lo
};

template <int NP>
struct Smem {
  __align__(128) unsigned char W[2][2][W_TILE];    // [branch][hi | lo]
  Stage st[NSTAGE];
  float w2[2][64];
  float b2[2];
  __align__(16) float zrow[64];                    // a zero history row: what the producer threads of rows past the chunk's end read
  uint64_t stage_full[NSTAGE], stage_empty[NSTAGE], s_full[NSTAGE], a_full[2], a_empty[2], d_full[2], d_empty[2], pool_full[2], pool_empty[2], wbar;
  uint32_t tmem_base;
};

// TMEM columns
constexpr uint32_t COL_D = 0;          // 2 x 64   hid accumulators
constexpr uint32_t COL_A = 128;        // 2 x (64 hi + 64 lo)   operand rows, K = 128 bf16 = 64 columns per part
constexpr uint32_t COL_POOL = 384;     // 2 x 32   pooled^T partials (candidate + 8 * column quarter)
constexpr uint32_t TMEM_COLS = 512;



__device__ __forceinline__ void issue_stage(Stage& st, const float* __restrict__ rows, const float* __restrict__ e, int toff,
                                            const float* __restrict__ tpg, int H, int C, int b, int c0, int ncg, int h0, int hl) {
  const int lane = threadIdx.x & 31;
  const float* src = rows + ((long long)b * H + h0) * 64;
  for (int i = lane; i < hl * 16; i += 32) cp_async16(&st.hf[(i >> 4) * HF_STRIDE + 4 * (i & 15)], src + 4 * i);
  for (int i = lane; i < ncg * 16; i += 32) {
    const int c = i >> 4, q = i & 15;
    const long long rc = (long long)b * C + c0 + c;
    cp_async16(&st.tv[c][4 * q], e + rc * E + toff + 4 * q);
    cp_async16(&st.tpv[c][4 * q], tpg + rc * 64 + 4 * q);
  }
  cp_async_commit();
}

// kScores: also store every valid row's fp32 score s[c][h] to scores [2][B][C][H] (nrm_forward_scores).  The four column-quarter
// partials of a row meet in shared memory behind sizeof(Smem<NP>) (SCORE_XCHG_BYTES more dynamic shared memory).  The kScores kernels
// are compiled in a translation unit of their own (nrm_attention_rs_scores.cu includes this file with NRM_RS_SCORES_TU defined):
// ptxas compiles a module as a whole, and any further kernel here changes the register assignment of the ones nrm_forward launches.
constexpr int SCORE_XCHG_BYTES = 2 * 3 * 128 * 4;    // [tile parity][column quarter 1..3][row of the tile]

template <int SPLIT, bool kScores>
__device__ __forceinline__ void attention_forward_rs(const float* __restrict__ pca32, const float* __restrict__ xhp, int B, int H, int C,
                                                     const unsigned char* __restrict__ img, const float* __restrict__ tp_all,
                                                     float* __restrict__ e, float* __restrict__ scores) {
  pdl_wait();
  pdl_trigger();
  constexpr int NP = SPLIT == 3 ? 2 : 1;
  constexpr int NT = SPLIT == 3 ? 3 : 1;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  Smem<NP>& sm = *reinterpret_cast<Smem<NP>*>(smem_raw);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

  // ---- prologue ---------------------------------------------------------------------------------------------------------------
  if (tid == 0) {
    for (int i = 0; i < NSTAGE; ++i) {
      umma::mbar_init(&sm.stage_full[i], 1);       // loader warp
      umma::mbar_init(&sm.stage_empty[i], N_PROD + 1);   // producer warps + the pooling product's commit
      umma::mbar_init(&sm.s_full[i], N_EPI);             // epilogue warps
    }
    for (int i = 0; i < 2; ++i) {
      umma::mbar_init(&sm.a_full[i], N_PROD);      // producer warps
      umma::mbar_init(&sm.a_empty[i], 1);          // commit of the hid product
      umma::mbar_init(&sm.d_full[i], 1);           // commit of the hid product
      umma::mbar_init(&sm.d_empty[i], N_EPI);      // epilogue warps
      umma::mbar_init(&sm.pool_full[i], 1);        // commit of the pooling product
      umma::mbar_init(&sm.pool_empty[i], 4);       // the 4 epilogue warps of column quarter 0
    }
    umma::mbar_init(&sm.wbar, 1);
    // weights of both branches: bulk copies by the TMA engine, under the rest of the prologue
    const uint32_t bar = umma::smem_u32(&sm.wbar);
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(bar), "r"(4u * W_TILE) : "memory");
    for (int br = 0; br < 2; ++br)
      for (int p = 0; p < 2; ++p)
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::"r"(umma::smem_u32(sm.W[br][p])),
                     "l"(img + (size_t)br * IMG_BRANCH_BYTES + (size_t)p * W_TILE), "r"(W_TILE), "r"(bar) : "memory");
  }
  if (tid < 128) {
    const int br = tid >> 6, j = tid & 63;
    const float* tail = reinterpret_cast<const float*>(img + (size_t)br * IMG_BRANCH_BYTES + 2 * W_TILE);
    sm.w2[br][j] = __ldg(tail + j);
    if (j == 0) sm.b2[br] = __ldg(tail + 64);
  }
  for (int i = tid; i < NSTAGE * 2 * 4096 / 4; i += THREADS) {     // score tiles start finite (stale entries meet zero history rows)
    const int s = i / (2 * 4096 / 4), r = i - s * (2 * 4096 / 4);
    reinterpret_cast<uint32_t*>(sm.st[s].s2[0])[r] = 0u;
  }
  if (tid < 64) sm.zrow[tid] = 0.f;
  if (warp == 0) umma::tmem_alloc(&sm.tmem_base, TMEM_COLS);
  umma::fence_async_smem();
  umma::fence_before_sync();
  __syncthreads();
  umma::fence_after_sync();
  const uint32_t tmem = sm.tmem_base;

  Geo g;
  g.B = B; g.H = H; g.C = C; g.G = (C + CG - 1) / CG; g.nchunks = (H + HCH - 1) / HCH;
  const long long U = 2LL * B * g.G;
  const int u0 = (int)(U * blockIdx.x / gridDim.x), u1 = (int)(U * (blockIdx.x + 1) / gridDim.x);
  const long long tp_branch = (long long)B * C * 64;

  if (warp == W_LOAD) {
    // =========================================== loader ===========================================
    RSPROF_TOTAL_BEGIN
    const int total = (u1 - u0) * g.nchunks;
    ChunkIter it_issue, it_fin;
    int n_issued = 0;
    auto issue = [&]() {
      const int s = n_issued % NSTAGE;
      RSPROF_WAIT(0, 0, umma::mbar_wait(&sm.stage_empty[s], ((n_issued / NSTAGE) & 1) ^ 1));
      const int br = it_issue.branch;
      issue_stage(sm.st[s], br == 0 ? xhp : pca32, e, br == 0 ? E_XT : E_PCAT, tp_all + br * tp_branch, H, C, it_issue.b, it_issue.c0,
                  it_issue.ncg, it_issue.h0, it_issue.hl);
      ++n_issued;
      if (n_issued < total) it_issue.next(g);
    };
    if (total > 0) { it_issue.set(g, u0, 0); it_fin.set(g, u0, 0); }
    while (n_issued < total && n_issued < NSTAGE - 1) issue();
    for (int k = 0; k < total; ++k) {
      RSPROF_WAIT(0, 1, if (n_issued - k - 1 >= 1) cp_async_wait<1>(); else cp_async_wait<0>());
      const int s = k % NSTAGE;
      arrive_warp(&sm.stage_full[s]);                    // every lane's copies have landed (wait_group above + the __syncwarp inside)
      if (k + 1 < total) it_fin.next(g);
      if (n_issued < total) issue();                     // into the stage chunk k - 1 used (its pooling product follows chunk k's first tile)
    }
    RSPROF_TOTAL_END(0);
  } else if (warp == W_MMA) {
    // =========================================== MMA issuer ===========================================
    if (umma::elect_one()) {
      umma::mbar_wait(&sm.wbar, 0);
      RSPROF_TOTAL_BEGIN
      constexpr uint32_t IDESC_HID = umma::make_idesc_bf16(128, 64);
      constexpr uint32_t IDESC_POOL = umma::make_idesc_bf16(64, 32, true, false);
      const uint64_t wdesc0 = umma::make_desc(umma::smem_u32(sm.W[0][0]), 1024, 128);      // + W_TILE / 16 per part, + 2 W_TILE / 16 per branch
      uint32_t chunk_seq = 0, tile_seq = 0, unit_seq = 0;
      // deferred pooling product of the previous chunk (issued after the next tile's hid product so that the tensor pipe
      // does not idle while the last epilogue of the chunk finishes)
      bool pend = false; uint32_t p_s = 0, p_ph = 0, p_ps = 0, p_pph = 0; bool p_first = false, p_last = false;
      auto do_pool = [&]() {
        RSPROF_WAIT(1, 2, umma::mbar_wait(&sm.s_full[p_s], p_ph));
        if (p_first) RSPROF_WAIT(1, 3, umma::mbar_wait(&sm.pool_empty[p_ps], p_pph ^ 1));
        umma::fence_after_sync();
        umma::mma_product<SPLIT, 4>(tmem + COL_POOL + 32 * p_ps, umma::op_tile64_mn(umma::smem_u32(sm.st[p_s].hbf[0])),
                                    umma::make_operand(umma::smem_u32(sm.st[p_s].s2[0]), 512, 128, 1024, 4096), IDESC_POOL, !p_first);
        umma::mma_commit(&sm.stage_empty[p_s]);
        if (p_last) umma::mma_commit(&sm.pool_full[p_ps]);
        pend = false;
      };
      for (int u = u0; u < u1; ++u, ++unit_seq) {
        int branch, b, c0, ncg; g.unit(u, branch, b, c0, ncg);
        for (int ci = 0; ci < g.nchunks; ++ci, ++chunk_seq) {
          int h0, hl, rows, ntiles; g.chunk(ci, ncg, h0, hl, rows, ntiles);
          for (int ti = 0; ti < ntiles; ++ti, ++tile_seq) {
            const uint32_t as = tile_seq & 1, aph = (tile_seq >> 1) & 1;
            RSPROF_WAIT(1, 0, umma::mbar_wait(&sm.a_full[as], aph));
            RSPROF_WAIT(1, 1, umma::mbar_wait(&sm.d_empty[as], aph ^ 1));
            umma::fence_after_sync();
            const uint32_t d = tmem + COL_D + 64 * as, a = tmem + COL_A + 128 * as;
#pragma unroll
            for (int t = 0; t < NT; ++t) {
              const uint32_t ap = (t == 2) ? 64u : 0u;
              const uint64_t wd = wdesc0 + (uint64_t)((2 * branch + (t == 1 ? 1 : 0)) * (W_TILE / 16));
#pragma unroll
              for (int ks = 0; ks < 8; ++ks) mma_bf16_ts(d, a + ap + 8 * ks, wd + (uint64_t)(ks * 128), IDESC_HID, (t > 0 || ks > 0) ? 1u : 0u);
            }
            umma::mma_commit(&sm.a_empty[as]);
            umma::mma_commit(&sm.d_full[as]);
            if (pend) do_pool();
          }
          pend = true; p_s = chunk_seq % NSTAGE; p_ph = (chunk_seq / NSTAGE) & 1; p_ps = unit_seq & 1; p_pph = (unit_seq >> 1) & 1;
          p_first = ci == 0; p_last = ci == g.nchunks - 1;
        }
      }
      if (pend) do_pool();
      RSPROF_TOTAL_END(1);
    }
  } else if (warp < W_EPI) {
    // =========================================== producers ===========================================
    RSPROF_TOTAL_BEGIN
    const uint32_t lane_sel = (uint32_t)(32 * (warp & 3)) << 16;
    uint32_t chunk_seq = 0, tile_seq = 0;
    for (int u = u0; u < u1; ++u) {
      int branch, b, c0, ncg; g.unit(u, branch, b, c0, ncg);
      for (int ci = 0; ci < g.nchunks; ++ci, ++chunk_seq) {
        int h0, hl, rows, ntiles; g.chunk(ci, ncg, h0, hl, rows, ntiles);
        const uint32_t s = chunk_seq % NSTAGE, ph = (chunk_seq / NSTAGE) & 1;
        const Stage& st = sm.st[s];
        const float inv_hl = 1.0f / (float)hl;
        RSPROF_WAIT(2, 0, umma::mbar_wait(&sm.stage_full[s], ph));
        for (int ti = 0; ti < ntiles; ++ti, ++tile_seq) {
          const uint32_t as = tile_seq & 1, aph = (tile_seq >> 1) & 1;
          RSPROF_WAIT(2, 1, umma::mbar_wait(&sm.a_empty[as], aph ^ 1));
          umma::fence_after_sync();
          const int rg = ti * 128 + 32 * (warp & 3) + lane;
          const bool valid = rg < rows;
          const int cl = valid ? __float2int_rz(((float)rg + 0.5f) * inv_hl) : 0, hloc = valid ? rg - cl * hl : 0;   // exact: rg < 640, hl <= 64
          const uint32_t a_hi = tmem + COL_A + 128 * as + lane_sel, a_lo = a_hi + 64;
          const float* hrow = valid ? &st.hf[hloc * HF_STRIDE] : sm.zrow;       // rows past the end: zero operand row, no selects
          const float* trow = &st.tv[cl][0];
          // The rows of the chunk's first candidate (cl == 0) cover every history row once: those threads also publish their
          // h half (bf16 hi | lo) as the K-major tile the pooling product reads MN-major; rows the chunk does not have are zeroed
          // by the threads of tile 0 that sit at those row numbers.
          const bool own_h = valid && cl == 0;
          const int zr = (ti == 0 && rg < HCH && rg >= hl) ? rg : -1;
          unsigned char* hb_own = const_cast<unsigned char*>(st.hbf[0]) + (uint32_t)(hloc >> 3) * umma::TILE64_SBO + (uint32_t)(hloc & 7) * 16u;
          const int khalf = warp >> 2;                    // this warp's half of the K range: passes kp = 2 khalf, 2 khalf + 1
#pragma unroll
          for (int kq = 0; kq < 2; ++kq) {                // two 8-column blocks (16 k) per pass
            const int kp = 2 * khalf + kq;
            uint32_t ph_hi[8], ph_lo[8], hh[8], hl_[8];
#pragma unroll
            for (int q = 0; q < 2; ++q) {
              const int kb = 2 * kp + q;
              const float4 h0v = *reinterpret_cast<const float4*>(hrow + 8 * kb), h1v = *reinterpret_cast<const float4*>(hrow + 8 * kb + 4);
              const float4 t0v = *reinterpret_cast<const float4*>(trow + 8 * kb), t1v = *reinterpret_cast<const float4*>(trow + 8 * kb + 4);
              const float hv[8] = {h0v.x, h0v.y, h0v.z, h0v.w, h1v.x, h1v.y, h1v.z, h1v.w};
              const float tv8[8] = {t0v.x, t0v.y, t0v.z, t0v.w, t1v.x, t1v.y, t1v.z, t1v.w};
#pragma unroll
              for (int i = 0; i < 4; ++i) {
                if (NP == 2) {
                  split2(hv[2 * i] * tv8[2 * i], hv[2 * i + 1] * tv8[2 * i + 1], ph_hi[4 * q + i], ph_lo[4 * q + i]);
                  split2(hv[2 * i], hv[2 * i + 1], hh[4 * q + i], hl_[4 * q + i]);
                } else {
                  ph_hi[4 * q + i] = pack_bf16(hv[2 * i] * tv8[2 * i], hv[2 * i + 1] * tv8[2 * i + 1]);
                  hh[4 * q + i] = pack_bf16(hv[2 * i], hv[2 * i + 1]);
                }
              }
              if (own_h) {
                *reinterpret_cast<uint4*>(hb_own + kb * umma::TILE64_LBO) = make_uint4(hh[4 * q], hh[4 * q + 1], hh[4 * q + 2], hh[4 * q + 3]);
                if (NP == 2) *reinterpret_cast<uint4*>(hb_own + 8192 + kb * umma::TILE64_LBO) = make_uint4(hl_[4 * q], hl_[4 * q + 1], hl_[4 * q + 2], hl_[4 * q + 3]);
              }
              if (zr >= 0) {
                unsigned char* z = const_cast<unsigned char*>(st.hbf[0]) + umma::tile64_offset(zr, kb);
                *reinterpret_cast<uint4*>(z) = make_uint4(0u, 0u, 0u, 0u);
                if (NP == 2) *reinterpret_cast<uint4*>(z + 8192) = make_uint4(0u, 0u, 0u, 0u);
              }
            }
            tmem_st8(a_hi + 8 * kp, ph_hi);               // k' = 16 kp .. 16 kp + 15  (t (.) h half)
            tmem_st8(a_hi + 32 + 8 * kp, hh);             // k' = 64 + 16 kp ..        (h half)
            if (NP == 2) { tmem_st8(a_lo + 8 * kp, ph_lo); tmem_st8(a_lo + 32 + 8 * kp, hl_); }
          }
          umma::fence_async_smem();                        // the h tile is read by the tensor core (async proxy) in the pooling product
          tmem_st_wait();
          umma::fence_before_sync();
          arrive_warp(&sm.a_full[as]);
        }
        arrive_warp(&sm.stage_empty[s]);                   // done with hf / tv / hbf of this stage
      }
    }
    if (warp == 0) RSPROF_TOTAL_END(2);
  } else {
    // =========================================== epilogue ===========================================
    RSPROF_TOTAL_BEGIN
    const int sp = warp & 3, cq = (warp - W_EPI) >> 2;     // TMEM sub-partition, quarter of the 64 hidden units
    const uint32_t lane_sel = (uint32_t)(32 * sp) << 16;
    uint32_t chunk_seq = 0, tile_seq = 0, unit_seq = 0;
    // deferred write-out of the previous unit's pooled vectors (its pooling product is issued one tile late)
    bool pend = false; uint32_t p_ps = 0, p_pph = 0; int p_branch = 0, p_b = 0, p_c0 = 0, p_ncg = 0;
    auto write_pooled = [&]() {
      if (cq == 0) {
        RSPROF_WAIT(3, 2, umma::mbar_wait(&sm.pool_full[p_ps], p_pph));
        umma::fence_after_sync();
        float v[32];
        umma::tmem_ld32(tmem + COL_POOL + 32 * p_ps + lane_sel, v);
        umma::fence_before_sync();
        arrive_warp(&sm.pool_empty[p_ps]);
        if (lane < 16) {                                   // an M = 64 accumulator occupies lanes 0-15 of each sub-partition: k = 16 sp + lane
          const int poff = p_branch == 0 ? E_LAB : E_TI;
          float* dst = e + ((long long)p_b * C + p_c0) * E + poff + 16 * sp + lane;
#pragma unroll
          for (int c = 0; c < CG; ++c)
            if (c < p_ncg) dst[(long long)c * E] = (v[c] + v[c + 8]) + (v[c + 16] + v[c + 24]);
        }
      }
      pend = false;
    };
    for (int u = u0; u < u1; ++u, ++unit_seq) {
      int branch, b, c0, ncg; g.unit(u, branch, b, c0, ncg);
      const float b2 = sm.b2[branch];
      f32x2 w2p[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) w2p[i] = pk(sm.w2[branch][16 * cq + 2 * i], sm.w2[branch][16 * cq + 2 * i + 1]);
      for (int ci = 0; ci < g.nchunks; ++ci, ++chunk_seq) {
        int h0, hl, rows, ntiles; g.chunk(ci, ncg, h0, hl, rows, ntiles);
        const uint32_t s = chunk_seq % NSTAGE, ph = (chunk_seq / NSTAGE) & 1;
        Stage& st = sm.st[s];
        const float inv_hl = 1.0f / (float)hl;
        RSPROF_WAIT(3, 0, umma::mbar_wait(&sm.stage_full[s], ph));
        for (int ti = 0; ti < ntiles; ++ti, ++tile_seq) {
          const uint32_t ds = tile_seq & 1, dph = (tile_seq >> 1) & 1;
          RSPROF_WAIT(3, 1, umma::mbar_wait(&sm.d_full[ds], dph));
          umma::fence_after_sync();
          float x[16];
          umma::tmem_ld16(tmem + COL_D + 64 * ds + 16 * cq + lane_sel, x);
          umma::fence_before_sync();
          arrive_warp(&sm.d_empty[ds]);                    // accumulator stage free: the next hid product may start
          const int rg = ti * 128 + 32 * sp + lane;
          const bool valid = rg < rows;
          const int cl = valid ? __float2int_rz(((float)rg + 0.5f) * inv_hl) : 0, hloc = valid ? rg - cl * hl : 0;
          const float* tp = &st.tpv[cl][16 * cq];
          // Exact-erf GELU (nrm_common.cuh: gelu_f; Abramowitz-Stegun 7.1.26) on the 16 hidden units of this thread, as 8 packed
          // pairs (fma.rn.f32x2: one issue slot per two FP32 operations -- the kernel is bound by issue slots) and written stage by
          // stage so that the independent dependency chains interleave.   With half = 0.5 erfc(|x| / sqrt 2) = poly(t) exp(-x^2 / 2):
          //     gelu(x) = x / 2 + |x| (1/2 - half)
          f32x2 xp[8], q[8];
#pragma unroll
          for (int j4 = 0; j4 < 4; ++j4) {
            const float4 t4 = *reinterpret_cast<const float4*>(tp + 4 * j4);
            xp[2 * j4] = add2(pk(x[4 * j4], x[4 * j4 + 1]), pk(t4.x, t4.y));
            xp[2 * j4 + 1] = add2(pk(x[4 * j4 + 2], x[4 * j4 + 3]), pk(t4.z, t4.w));
          }
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            float a, b, ta, tb, ea, eb;
            upk(xp[i], a, b);
            asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(ta) : "f"(fmaf(fabsf(a), 0.23164189f, 1.0f)));      // t = 1 / (1 + 0.3275911 |x| / sqrt 2)
            asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(tb) : "f"(fmaf(fabsf(b), 0.23164189f, 1.0f)));
            f32x2 ar = mul2(mul2(xp[i], xp[i]), pk(-0.72134752044448170368f, -0.72134752044448170368f));   // -x^2 log2(e) / 2
            upk(ar, ea, eb);
            asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(ea) : "f"(ea));
            asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(eb) : "f"(eb));
            const f32x2 t2 = pk(ta, tb);
            f32x2 poly = fma2(t2, pk(0.5f * 1.061405429f, 0.5f * 1.061405429f), pk(0.5f * -1.453152027f, 0.5f * -1.453152027f));
            poly = fma2(t2, poly, pk(0.5f * 1.421413741f, 0.5f * 1.421413741f));
            poly = fma2(t2, poly, pk(0.5f * -0.284496736f, 0.5f * -0.284496736f));
            poly = fma2(t2, poly, pk(0.5f * 0.254829592f, 0.5f * 0.254829592f));
            poly = mul2(poly, t2);                                                                           // 0.5 erfc(z) / exp(-z^2)
            q[i] = fma2(poly, mul2(pk(ea, eb), pk(-1.f, -1.f)), pk(0.5f, 0.5f));                             // 1/2 - half
          }
          f32x2 acc2 = pk(cq == 0 ? b2 : 0.f, 0.f);
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            float a, b, qa, qb, ha, hb;
            upk(xp[i], a, b);
            upk(q[i], qa, qb);
            upk(mul2(xp[i], pk(0.5f, 0.5f)), ha, hb);
            const float g0 = fmaf(fabsf(a), qa, ha), g1 = fmaf(fabsf(b), qb, hb);
            acc2 = fma2(pk(g0, g1), w2p[i], acc2);
          }
          float acc, acc_hi;
          upk(acc2, acc, acc_hi);
          acc += acc_hi;
          if (valid) {
            const int slot = cl + 8 * cq;
            const uint32_t off = (uint32_t)(hloc >> 3) * 512u + (uint32_t)(slot >> 3) * 128u + (uint32_t)(slot & 7) * 16u + (uint32_t)(hloc & 7) * 2u;
            const __nv_bfloat16 hi = __float2bfloat16_rn(acc);
            *reinterpret_cast<__nv_bfloat16*>(st.s2[0] + off) = hi;
            if (NP == 2) *reinterpret_cast<__nv_bfloat16*>(st.s2[1] + off) = __float2bfloat16_rn(acc - __bfloat162float(hi));
          }
          if constexpr (kScores) {
            // s = (quarter 0 + quarter 1) + (quarter 2 + quarter 3), each quarter's partial as the epilogue computed it (fp32, before
            // the bf16 split).  The four warps of sub-partition sp meet at named barrier 1 + sp; the exchange slots alternate with the
            // tile parity, and a warp cannot overwrite a slot before quarter 0 has passed the NEXT barrier, i.e. read this one.
            float* xchg = reinterpret_cast<float*>(smem_raw + sizeof(Smem<NP>)) + (tile_seq & 1) * (3 * 128) + 32 * sp + lane;
            if (cq > 0) xchg[(cq - 1) * 128] = acc;
            __syncwarp();                                  // bar.sync is the ALIGNED barrier: the warp must arrive converged
            asm volatile("bar.sync %0, 128;\n" ::"r"(1 + sp) : "memory");
            if (cq == 0 && valid)
              scores[(((long long)branch * B + b) * C + c0 + cl) * H + h0 + hloc] = (acc + xchg[0]) + (xchg[128] + xchg[256]);
          }
          if (ti == ntiles - 1) {
            umma::fence_async_smem();                      // scores are read by the tensor core (async proxy)
            arrive_warp(&sm.s_full[s]);
          }
          if (pend) write_pooled();
        }
      }
      pend = true; p_ps = unit_seq & 1; p_pph = (unit_seq >> 1) & 1; p_branch = branch; p_b = b; p_c0 = c0; p_ncg = ncg;
    }
    if (pend) write_pooled();
    if (warp == W_EPI) RSPROF_TOTAL_END(3);
  }

  umma::fence_before_sync();
  __syncthreads();
  if (warp == 0) umma::tmem_dealloc(tmem, TMEM_COLS);
}

#ifndef NRM_RS_SCORES_TU
template <int SPLIT>
__global__ void __launch_bounds__(THREADS, 1)
attention_forward_rs_kernel(const float* __restrict__ pca32, const float* __restrict__ xhp, int B, int H, int C,
                            const unsigned char* __restrict__ img, const float* __restrict__ tp_all, float* __restrict__ e) {
  attention_forward_rs<SPLIT, false>(pca32, xhp, B, H, C, img, tp_all, e, nullptr);
}
#else
template <int SPLIT>
__global__ void __launch_bounds__(THREADS, 1)
attention_forward_rs_scores_kernel(const float* __restrict__ pca32, const float* __restrict__ xhp, int B, int H, int C,
                                   const unsigned char* __restrict__ img, const float* __restrict__ tp_all, float* __restrict__ e,
                                   float* __restrict__ scores) {
  attention_forward_rs<SPLIT, true>(pca32, xhp, B, H, C, img, tp_all, e, scores);
}
#endif

}  // namespace rs

#ifndef NRM_RS_SCORES_TU
int launch_attention_prep_rs(const float* P, Workspace& w, cudaStream_t s) {
  launch_pdl(rs::att_prep_rs_kernel, dim3(8, 2), dim3(256), 0, s, P, reinterpret_cast<unsigned char*>(w.att_rs_img));
  NRM_LAUNCH_CHECK("att_prep_rs_kernel");
  return NRM_OK;
}

template <int SPLIT>
static int launch_fwd_rs(const BatchPtrs& in, Workspace& w, cudaStream_t s) {
  constexpr int NP = SPLIT == 3 ? 2 : 1;
  const size_t smem = sizeof(rs::Smem<NP>);
  const long long G = (w.C + rs::CG - 1) / rs::CG, U = 2LL * w.B * G;
  const int grid = (int)min(U, (long long)sm_count());
  NRM_CUDA(cudaFuncSetAttribute(rs::attention_forward_rs_kernel<SPLIT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  launch_pdl(rs::attention_forward_rs_kernel<SPLIT>, dim3(grid), dim3(rs::THREADS), smem, s, w.pca_h, w.xh, w.B, w.H, w.C,
             reinterpret_cast<const unsigned char*>(w.att_rs_img), w.tp, w.e);
  NRM_LAUNCH_CHECK("attention_forward_rs_kernel");
  return NRM_OK;
}

// both branches in one launch; w.scores non-null: the score-exporting kernels (nrm_attention_rs_scores.cu)
int launch_attention_forward_rs(const BatchPtrs& in, Workspace& w, int precision, cudaStream_t s) {
  if (w.scores != nullptr) return launch_attention_forward_rs_scores(w, precision, s);
  return precision == NRM_PRECISION_BF16 ? launch_fwd_rs<1>(in, w, s) : launch_fwd_rs<3>(in, w, s);
}

size_t attention_rs_image_bytes() { return (size_t)rs::img_bytes(); }

int rsprof_read(long long* host_out64) {
#ifdef NRM_RS_PROFILE
  long long zero[64] = {0};
  NRM_CUDA(cudaDeviceSynchronize());
  NRM_CUDA(cudaMemcpyFromSymbol(host_out64, rs::g_rsprof, sizeof(zero)));
  NRM_CUDA(cudaMemcpyToSymbol(rs::g_rsprof, zero, sizeof(zero)));
  return NRM_OK;
#else
  (void)host_out64;
  set_error("library built without -DNRM_RS_PROFILE");
  return NRM_EUNSUPPORTED;
#endif
}

#else
template <int SPLIT>
static int launch_fwd_rs_scores(Workspace& w, cudaStream_t s) {
  constexpr int NP = SPLIT == 3 ? 2 : 1;
  const size_t smem = sizeof(rs::Smem<NP>) + rs::SCORE_XCHG_BYTES;
  const long long G = (w.C + rs::CG - 1) / rs::CG, U = 2LL * w.B * G;
  const int grid = (int)min(U, (long long)sm_count());
  NRM_CUDA(cudaFuncSetAttribute(rs::attention_forward_rs_scores_kernel<SPLIT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  launch_pdl(rs::attention_forward_rs_scores_kernel<SPLIT>, dim3(grid), dim3(rs::THREADS), smem, s, w.pca_h, w.xh, w.B, w.H, w.C,
             reinterpret_cast<const unsigned char*>(w.att_rs_img), w.tp, w.e, w.scores);
  NRM_LAUNCH_CHECK("attention_forward_rs_scores_kernel");
  return NRM_OK;
}

int launch_attention_forward_rs_scores(Workspace& w, int precision, cudaStream_t s) {
  return precision == NRM_PRECISION_BF16 ? launch_fwd_rs_scores<1>(w, s) : launch_fwd_rs_scores<3>(w, s);
}
#endif

}  // namespace nrm
