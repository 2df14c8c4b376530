// Pairwise (candidate x history) MLP attention + sum pooling, forward and backward,
// fp32 CUDA-core path.  Reference: PointwiseAttentionExpanded.forward
// (models/attention_model.py:52-97) and the pooling at
// models/user_invariant_interest_model.py:83-87.
//
// Reduced form (DESIGN.md section 3; checked against autograd in tests/test_reduced_algebra.py):
// with fc1.weight = [Wa|Wb|Wc|Wd] over the concat [h, t, t-h, t*h],
//     hid[c,h,:] = W_c h + tp_c,   W_c = Wd diag(t_c) + (Wa - Wc),   tp_c = (Wb + Wc) t_c + b1
//     s[c,h]     = w2 . gelu(hid[c,h,:]) + b2,        pooled[c,:] = sum_h s[c,h] h[h,:]
// so one candidate's hidden tile is a 64(h) x 64(j) x 64(k) GEMM of the staged history tile
// with a per-candidate matrix built in shared memory; the [B,C,H,256] concat never exists.
//
// One CTA works on one impression at a time: its history is staged once per 64-row tile
// (row-major for pooling / dW products, k-major for the hidden GEMM) and reused by all C
// candidates.  History rows past H are zero-filled, which makes them inert everywhere.
#include "nrm_kernels.cuh"

namespace nrm {

constexpr int HT = 64;      // history rows per tile
constexpr int CCH = 8;      // candidates per chunk
constexpr int WS = 65;      // row stride of the row-major 64x64 weight blocks (conflict-free both ways)
constexpr int TS = 68;      // row stride of k-major tiles (keeps float4 alignment)
constexpr int ATT_THREADS = 256;

struct AttSmemFwd {
  float Wd[64 * WS], A[64 * WS], Bm[64 * WS];
  float b1[64], w2[64];
  float h[HT * 64];          // [row][k]
  float hT[64 * TS];         // [k][row]
  float WcT[64 * TS];        // [k][j]
  float t[CCH * 64], tp[CCH * 64], s[CCH * HT];
};

struct AttSmemBwd {
  float Wd[64 * WS], A[64 * WS], Bm[64 * WS];
  float b1[64], w2[64];
  float h[HT * 64];
  float hT[64 * TS];
  float WcT[64 * TS];        // [k][j]
  float Wc[64 * 64];         // [j][k]
  float dhid[HT * 64];       // [row][j]
  float dhidT[64 * TS];      // [j][row]
  float dA[64 * 64], dWd[64 * 64], dBm[64 * 64];   // per-CTA accumulators [j][k]
  float t[CCH * 64], tp[CCH * 64], dP[CCH * 64], ds[CCH * HT], s[CCH * HT];
  float Gt[64];
  float gpart[16 * 64];      // per row-group partial sums of dhid columns; reused for the final dw2/db2 reduce
  float dtpart[16 * 64];
};

// fc1.weight [64,256] -> row-major blocks A = Wa - Wc, Bm = Wb + Wc, Wd (stride WS); fc1.bias, fc2.weight
__device__ __forceinline__ void load_att_weights(const float* __restrict__ P, AttOffsets off, float* Wd, float* A,
                                                 float* Bm, float* b1, float* w2) {
  const float* W = P + off.fc1_w;
  for (int i = threadIdx.x; i < 64 * 64; i += ATT_THREADS) {
    const int j = i >> 6, k = i & 63;
    const float wa = __ldg(W + j * 256 + k), wb = __ldg(W + j * 256 + 64 + k);
    const float wc = __ldg(W + j * 256 + 128 + k), wd = __ldg(W + j * 256 + 192 + k);
    A[j * WS + k] = wa - wc;
    Bm[j * WS + k] = wb + wc;
    Wd[j * WS + k] = wd;
  }
  if (threadIdx.x < 64) {
    b1[threadIdx.x] = __ldg(P + off.fc1_b + threadIdx.x);
    w2[threadIdx.x] = __ldg(P + off.fc2_w + threadIdx.x);
  }
}

// Stage history rows [r0, r0+64) of impression b: h[row][k] and hT[k][row]; rows >= H are zero.
template <int BRANCH>
__device__ __forceinline__ void load_history_tile(const double* __restrict__ xh, const float* __restrict__ xhp,
                                                  long long b, int H, int r0, float* h, float* hT) {
  if (BRANCH == 0) {
    // w1-projected label features, fp32 [NH,64]
    for (int f = threadIdx.x; f < HT * 16; f += ATT_THREADS) {
      const int row = f >> 4, k4 = f & 15;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (r0 + row < H) v = __ldg(reinterpret_cast<const float4*>(xhp + (b * H + r0 + row) * 64) + k4);
      *reinterpret_cast<float4*>(h + row * 64 + 4 * k4) = v;
      hT[(4 * k4 + 0) * TS + row] = v.x; hT[(4 * k4 + 1) * TS + row] = v.y;
      hT[(4 * k4 + 2) * TS + row] = v.z; hT[(4 * k4 + 3) * TS + row] = v.w;
    }
  } else {
    // PCA columns 4..67 of the packed float64 rows, converted in registers
    for (int f = threadIdx.x; f < HT * 32; f += ATT_THREADS) {
      const int row = f >> 5, k2 = f & 31;
      double2 v = make_double2(0.0, 0.0);
      if (r0 + row < H) v = __ldg(reinterpret_cast<const double2*>(xh + (b * H + r0 + row) * HC + 4) + k2);
      const float a = (float)v.x, c = (float)v.y;
      *reinterpret_cast<float2*>(h + row * 64 + 2 * k2) = make_float2(a, c);
      hT[(2 * k2 + 0) * TS + row] = a; hT[(2 * k2 + 1) * TS + row] = c;
    }
  }
}

// WcT[k][j] = Wd[j][k] * t[k] + A[j][k]
__device__ __forceinline__ void build_WcT(const float* Wd, const float* A, const float* t, float* WcT) {
  const int j = threadIdx.x & 63;
#pragma unroll 4
  for (int k = threadIdx.x >> 6; k < 64; k += 4) WcT[k * TS + j] = fmaf(Wd[j * WS + k], t[k], A[j * WS + k]);
}
// Wc[j][k], row-major
__device__ __forceinline__ void build_Wc(const float* Wd, const float* A, const float* t, float* Wc) {
  const int k = threadIdx.x & 63;
  const float tk = t[k];
#pragma unroll 4
  for (int j = threadIdx.x >> 6; j < 64; j += 4) Wc[j * 64 + k] = fmaf(Wd[j * WS + k], tk, A[j * WS + k]);
}

// acc[r][jj] = sum_k hT[k][4tr + r] * WcT[k][4tc + jj]
__device__ __forceinline__ void hidden_gemm(const float* hT, const float* WcT, int tr, int tc, float acc[4][4]) {
#pragma unroll
  for (int r = 0; r < 4; ++r)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[r][j] = 0.f;
#pragma unroll 8
  for (int k = 0; k < 64; ++k) {
    const float4 a = *reinterpret_cast<const float4*>(hT + k * TS + 4 * tr);
    const float4 b = *reinterpret_cast<const float4*>(WcT + k * TS + 4 * tc);
    const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
    for (int r = 0; r < 4; ++r)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[r][j] = fmaf(av[r], bv[j], acc[r][j]);
  }
}

__device__ __forceinline__ float reduce16(float v) {   // sum over the 16 lanes that share tr
  v += __shfl_xor_sync(0xffffffffu, v, 8);
  v += __shfl_xor_sync(0xffffffffu, v, 4);
  v += __shfl_xor_sync(0xffffffffu, v, 2);
  v += __shfl_xor_sync(0xffffffffu, v, 1);
  return v;
}

// ---------------------------------------------------------------------------------
// forward: grid = B (one impression per CTA), 256 threads, ~108 KB shared
// ---------------------------------------------------------------------------------
// kScores: also store every valid row's score s[c][h] to scores [2][B][C][H] (nrm_forward_scores); with kScores = false the kernel
// is the one nrm_forward has always launched.
template <int BRANCH, bool kScores>
__global__ void __launch_bounds__(ATT_THREADS, 2)
attention_forward_kernel(const double* __restrict__ xh, const float* __restrict__ xhp, int B, int H, int C,
                         const float* __restrict__ P, float* __restrict__ e, float* __restrict__ scores) {
  pdl_wait();                                          // programmatic dependent launch: see nrm_common.cuh
  pdl_trigger();
  extern __shared__ __align__(16) unsigned char smem_raw[];
  AttSmemFwd& sm = *reinterpret_cast<AttSmemFwd*>(smem_raw);
  constexpr AttOffsets off = BRANCH == 0 ? ATT_LABEL : ATT_TI;
  constexpr int TOFF = BRANCH == 0 ? E_XT : E_PCAT;     // candidate vectors inside e_concat
  constexpr int POFF = BRANCH == 0 ? E_LAB : E_TI;      // pooled output inside e_concat
  const int tid = threadIdx.x, tr = tid >> 4, tc = tid & 15;
  load_att_weights(P, off, sm.Wd, sm.A, sm.Bm, sm.b1, sm.w2);
  const float b2 = __ldg(P + off.fc2_b);

  for (long long b = blockIdx.x; b < B; b += gridDim.x) {
    for (int r0 = 0; r0 < H; r0 += HT) {
      __syncthreads();
      load_history_tile<BRANCH>(xh, xhp, b, H, r0, sm.h, sm.hT);
      for (int c0 = 0; c0 < C; c0 += CCH) {
        const int nc = min(CCH, C - c0);
        __syncthreads();
        for (int i = tid; i < nc * 64; i += ATT_THREADS)
          sm.t[i] = e[((b * C + c0 + (i >> 6)) * E) + TOFF + (i & 63)];
        __syncthreads();
        for (int i = tid; i < nc * 64; i += ATT_THREADS) {
          const int cl = i >> 6, j = i & 63;
          float v = sm.b1[j];
#pragma unroll 8
          for (int k = 0; k < 64; ++k) v = fmaf(sm.Bm[j * WS + k], sm.t[cl * 64 + k], v);
          sm.tp[i] = v;
        }
        for (int cl = 0; cl < nc; ++cl) {
          __syncthreads();
          build_WcT(sm.Wd, sm.A, sm.t + cl * 64, sm.WcT);
          __syncthreads();
          float acc[4][4];
          hidden_gemm(sm.hT, sm.WcT, tr, tc, acc);
          float tpv[4], w2v[4];
#pragma unroll
          for (int j = 0; j < 4; ++j) { tpv[j] = sm.tp[cl * 64 + 4 * tc + j]; w2v[j] = sm.w2[4 * tc + j]; }
#pragma unroll
          for (int r = 0; r < 4; ++r) {
            float part = 0.f;
#pragma unroll
            for (int j = 0; j < 4; ++j) part = fmaf(gelu_f(acc[r][j] + tpv[j]), w2v[j], part);
            part = reduce16(part);
            if (tc == 0) sm.s[cl * HT + 4 * tr + r] = part + b2;
            if (kScores && tc == 0 && r0 + 4 * tr + r < H)
              scores[((BRANCH * (long long)B + b) * C + c0 + cl) * H + r0 + 4 * tr + r] = part + b2;
          }
        }
        __syncthreads();
        // pooled[c][k] (+)= sum_row s[c][row] * h[row][k]
        for (int i = tid; i < nc * 64; i += ATT_THREADS) {
          const int cl = i >> 6, k = i & 63;
          float v = 0.f;
#pragma unroll 8
          for (int row = 0; row < HT; ++row) v = fmaf(sm.s[cl * HT + row], sm.h[row * 64 + k], v);
          float* dst = e + ((b * C + c0 + cl) * E) + POFF + k;
          if (r0 == 0) *dst = v; else *dst += v;
        }
      }
    }
  }
}

// ---------------------------------------------------------------------------------
// backward: persistent grid (<= 148 CTAs), 256 threads, ~203 KB shared.
// Recomputes the hidden tile, then per candidate:
//   dhid = ds w2 gelu'(hid);  Gt = sum_h dhid;  S = dhid^T h;
//   dA += S; dWd += S diag(t); dBm += Gt t^T; db1 += Gt;
//   dt = Gt Bm + sum_j S.Wd;  dh += dhid W_c   (dt, dh: label only)
// Per-CTA partial sums of dA, dWd, dBm, db1, dfc2 go to part[blockIdx.x].
// ---------------------------------------------------------------------------------
template <int BRANCH>
__global__ void __launch_bounds__(ATT_THREADS, 1)
attention_backward_kernel(const double* __restrict__ xh, const float* __restrict__ xhp, int B, int H, int C,
                          const float* __restrict__ P, const float* __restrict__ e, const float* __restrict__ de,
                          float* __restrict__ dxh, float* __restrict__ dxt, float* __restrict__ part) {
  pdl_wait();                                          // programmatic dependent launch: see nrm_common.cuh
  pdl_trigger();
  extern __shared__ __align__(16) unsigned char smem_raw[];
  AttSmemBwd& sm = *reinterpret_cast<AttSmemBwd*>(smem_raw);
  constexpr AttOffsets off = BRANCH == 0 ? ATT_LABEL : ATT_TI;
  constexpr int TOFF = BRANCH == 0 ? E_XT : E_PCAT;
  constexpr int POFF = BRANCH == 0 ? E_LAB : E_TI;
  constexpr bool INPUT_GRADS = (BRANCH == 0);
  const int tid = threadIdx.x, tr = tid >> 4, tc = tid & 15;
  load_att_weights(P, off, sm.Wd, sm.A, sm.Bm, sm.b1, sm.w2);
  for (int i = tid; i < 64 * 64; i += ATT_THREADS) { sm.dA[i] = 0.f; sm.dWd[i] = 0.f; sm.dBm[i] = 0.f; }
  const float b2 = __ldg(P + off.fc2_b);
  float dw2_acc[4] = {0.f, 0.f, 0.f, 0.f};
  float db1_acc[4] = {0.f, 0.f, 0.f, 0.f};      // only the tc == 0 lane of each row group keeps these
  float db2_acc = 0.f;

  for (long long b = blockIdx.x; b < B; b += gridDim.x) {
    for (int r0 = 0; r0 < H; r0 += HT) {
      __syncthreads();
      load_history_tile<BRANCH>(xh, xhp, b, H, r0, sm.h, sm.hT);
      float dhacc[4][4];
#pragma unroll
      for (int r = 0; r < 4; ++r)
#pragma unroll
        for (int k = 0; k < 4; ++k) dhacc[r][k] = 0.f;

      for (int c0 = 0; c0 < C; c0 += CCH) {
        const int nc = min(CCH, C - c0);
        __syncthreads();
        for (int i = tid; i < nc * 64; i += ATT_THREADS) {
          const long long rowc = (b * C + c0 + (i >> 6)) * E;
          sm.t[i] = e[rowc + TOFF + (i & 63)];
          sm.dP[i] = de[rowc + POFF + (i & 63)];
        }
        __syncthreads();
        for (int i = tid; i < nc * 64; i += ATT_THREADS) {
          const int cl = i >> 6, j = i & 63;      // j doubles as the history row for ds
          float v = sm.b1[j], d = 0.f;
#pragma unroll 8
          for (int k = 0; k < 64; ++k) {
            v = fmaf(sm.Bm[j * WS + k], sm.t[cl * 64 + k], v);
            d = fmaf(sm.dP[cl * 64 + k], sm.hT[k * TS + j], d);
          }
          sm.tp[i] = v;
          sm.ds[cl * HT + j] = d;
        }
        for (int cl = 0; cl < nc; ++cl) {
          const long long rc = b * C + c0 + cl;
          __syncthreads();                                   // (a) previous candidate fully consumed
          build_WcT(sm.Wd, sm.A, sm.t + cl * 64, sm.WcT);
          if (INPUT_GRADS) build_Wc(sm.Wd, sm.A, sm.t + cl * 64, sm.Wc);
          __syncthreads();                                   // (b)
          float acc[4][4];
          hidden_gemm(sm.hT, sm.WcT, tr, tc, acc);
          {
            float tpv[4], w2v[4], gsum[4] = {0.f, 0.f, 0.f, 0.f};
            float dhv[4][4];
#pragma unroll
            for (int j = 0; j < 4; ++j) { tpv[j] = sm.tp[cl * 64 + 4 * tc + j]; w2v[j] = sm.w2[4 * tc + j]; }
#pragma unroll
            for (int r = 0; r < 4; ++r) {
              const float dsr = sm.ds[cl * HT + 4 * tr + r];
              float spart = 0.f;
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                float gp;
                const float g = gelu_both(acc[r][j] + tpv[j], gp);
                spart = fmaf(g, w2v[j], spart);
                dw2_acc[j] = fmaf(dsr, g, dw2_acc[j]);
                const float dh = dsr * w2v[j] * gp;
                dhv[r][j] = dh;
                gsum[j] += dh;
              }
              if (INPUT_GRADS) {
                spart = reduce16(spart);
                if (tc == 0) sm.s[cl * HT + 4 * tr + r] = spart + b2;
              }
              if (tc == 0) db2_acc += dsr;
              *reinterpret_cast<float4*>(sm.dhid + (4 * tr + r) * 64 + 4 * tc) =
                  make_float4(dhv[r][0], dhv[r][1], dhv[r][2], dhv[r][3]);
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              if (INPUT_GRADS)
                *reinterpret_cast<float4*>(sm.dhidT + (4 * tc + j) * TS + 4 * tr) =
                    make_float4(dhv[0][j], dhv[1][j], dhv[2][j], dhv[3][j]);
              sm.gpart[tr * 64 + 4 * tc + j] = gsum[j];
            }
          }
          __syncthreads();                                   // (c) dhid, dhidT, gpart visible
          if (INPUT_GRADS && tid < 64) {
            float g = 0.f;
#pragma unroll
            for (int q = 0; q < 16; ++q) g += sm.gpart[q * 64 + tid];
            sm.Gt[tid] = g;
          }
          {
            // Gt[j] = sum_h dhid[h][j] for this thread's four j (= 4tr..4tr+3)
            float4 g4 = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int q = 0; q < 16; ++q) {
              const float4 v = *reinterpret_cast<const float4*>(sm.gpart + q * 64 + 4 * tr);
              g4.x += v.x; g4.y += v.y; g4.z += v.z; g4.w += v.w;
            }
            const float gv[4] = {g4.x, g4.y, g4.z, g4.w};
            const float4 tq0 = *reinterpret_cast<const float4*>(sm.t + cl * 64 + 4 * tc);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              float4* pb = reinterpret_cast<float4*>(sm.dBm + (4 * tr + j) * 64 + 4 * tc);
              float4 vb = *pb;
              vb.x = fmaf(gv[j], tq0.x, vb.x); vb.y = fmaf(gv[j], tq0.y, vb.y);
              vb.z = fmaf(gv[j], tq0.z, vb.z); vb.w = fmaf(gv[j], tq0.w, vb.w);
              *pb = vb;
              if (tc == 0) db1_acc[j] += gv[j];
            }
          }
          {
            // S[jj][kk] = sum_row dhid[row][4tr+jj] * h[row][4tc+kk]   (here tr indexes j, tc indexes k)
            float S[4][4];
#pragma unroll
            for (int j = 0; j < 4; ++j)
#pragma unroll
              for (int k = 0; k < 4; ++k) S[j][k] = 0.f;
#pragma unroll 8
            for (int row = 0; row < HT; ++row) {
              const float4 a = *reinterpret_cast<const float4*>(sm.dhid + row * 64 + 4 * tr);
              const float4 bq = *reinterpret_cast<const float4*>(sm.h + row * 64 + 4 * tc);
              const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {bq.x, bq.y, bq.z, bq.w};
#pragma unroll
              for (int j = 0; j < 4; ++j)
#pragma unroll
                for (int k = 0; k < 4; ++k) S[j][k] = fmaf(av[j], bv[k], S[j][k]);
            }
            const float4 tq = *reinterpret_cast<const float4*>(sm.t + cl * 64 + 4 * tc);
            const float tv[4] = {tq.x, tq.y, tq.z, tq.w};
            float dtp[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              float4* pa = reinterpret_cast<float4*>(sm.dA + (4 * tr + j) * 64 + 4 * tc);
              float4* pd = reinterpret_cast<float4*>(sm.dWd + (4 * tr + j) * 64 + 4 * tc);
              float4 va = *pa, vd = *pd;
              va.x += S[j][0]; va.y += S[j][1]; va.z += S[j][2]; va.w += S[j][3];
              vd.x = fmaf(S[j][0], tv[0], vd.x); vd.y = fmaf(S[j][1], tv[1], vd.y);
              vd.z = fmaf(S[j][2], tv[2], vd.z); vd.w = fmaf(S[j][3], tv[3], vd.w);
              *pa = va; *pd = vd;
              if (INPUT_GRADS) {
#pragma unroll
                for (int k = 0; k < 4; ++k) dtp[k] = fmaf(S[j][k], sm.Wd[(4 * tr + j) * WS + 4 * tc + k], dtp[k]);
              }
            }
            if (INPUT_GRADS) {
#pragma unroll
              for (int k = 0; k < 4; ++k) sm.dtpart[tr * 64 + 4 * tc + k] = dtp[k];
            }
          }
          if (INPUT_GRADS) {
            // dhacc[r][kk] += sum_j dhidT[j][4tr+r] * Wc[j][4tc+kk]
#pragma unroll 8
            for (int j = 0; j < 64; ++j) {
              const float4 a = *reinterpret_cast<const float4*>(sm.dhidT + j * TS + 4 * tr);
              const float4 bq = *reinterpret_cast<const float4*>(sm.Wc + j * 64 + 4 * tc);
              const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {bq.x, bq.y, bq.z, bq.w};
#pragma unroll
              for (int r = 0; r < 4; ++r)
#pragma unroll
                for (int k = 0; k < 4; ++k) dhacc[r][k] = fmaf(av[r], bv[k], dhacc[r][k]);
            }
            __syncthreads();                                 // (d) dtpart, Gt visible
            if (tid < 64) {
              float d = 0.f;
#pragma unroll
              for (int q = 0; q < 16; ++q) d += sm.dtpart[q * 64 + tid];
#pragma unroll 8
              for (int j = 0; j < 64; ++j) d = fmaf(sm.Gt[j], sm.Bm[j * WS + tid], d);
              float* dst = dxt + rc * 64 + tid;
              if (r0 == 0) *dst = d + de[rc * E + E_XT + tid];   // + the direct ec path (user_model.py:31)
              else *dst += d;
            }
          }
        }
        if (INPUT_GRADS) {
          __syncthreads();                                   // s of the whole chunk visible
          // pooling path: dh[row][k] += sum_c s[c][row] * dP[c][k]
          for (int cl = 0; cl < nc; ++cl) {
            const float4 a = *reinterpret_cast<const float4*>(sm.s + cl * HT + 4 * tr);
            const float4 bq = *reinterpret_cast<const float4*>(sm.dP + cl * 64 + 4 * tc);
            const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {bq.x, bq.y, bq.z, bq.w};
#pragma unroll
            for (int r = 0; r < 4; ++r)
#pragma unroll
              for (int k = 0; k < 4; ++k) dhacc[r][k] = fmaf(av[r], bv[k], dhacc[r][k]);
          }
        }
      }
      if (INPUT_GRADS) {
#pragma unroll
        for (int r = 0; r < 4; ++r) {
          const int row = r0 + 4 * tr + r;
          if (row < H)
            *reinterpret_cast<float4*>(dxh + (b * H + row) * 64 + 4 * tc) =
                make_float4(dhacc[r][0], dhacc[r][1], dhacc[r][2], dhacc[r][3]);
        }
      }
    }
  }

  // ---- per-CTA partial sums -> part[blockIdx.x]
  __syncthreads();
  float* out = part + (long long)blockIdx.x * ATT_PARTIAL;
  for (int i = tid; i < 64 * 64; i += ATT_THREADS) {
    out[i] = sm.dA[i]; out[64 * 64 + i] = sm.dWd[i]; out[2 * 64 * 64 + i] = sm.dBm[i];
  }
  if (tc == 0) {
#pragma unroll
    for (int j = 0; j < 4; ++j) out[3 * 64 * 64 + 64 + 4 * tr + j] = db1_acc[j];
  }
#pragma unroll
  for (int j = 0; j < 4; ++j) sm.gpart[tr * 64 + 4 * tc + j] = dw2_acc[j];
  sm.dtpart[tid] = db2_acc;
  __syncthreads();
  if (tid < 64) {
    float g = 0.f;
#pragma unroll
    for (int q = 0; q < 16; ++q) g += sm.gpart[q * 64 + tid];
    out[3 * 64 * 64 + tid] = g;
  }
  if (tid == 0) {
    float d = 0.f;
    for (int q = 0; q < ATT_THREADS; q += 16) d += sm.dtpart[q];   // only tc == 0 lanes accumulated
    out[3 * 64 * 64 + 128] = d;
  }
}

// Sum the per-CTA partials in fixed order and scatter them into the flat gradient:
// fc1.weight grad [64,256] = [dA | dBm | dBm - dA | dWd]; fc1.bias = db1; fc2.weight = dw2; fc2.bias = db2.
__global__ void __launch_bounds__(256)
attention_compose_kernel(const float* __restrict__ part, int nparts, AttOffsets off, float* __restrict__ grads) {
  pdl_wait();                                          // programmatic dependent launch: see nrm_common.cuh
  pdl_trigger();
  // block = 64 consecutive (j,k) entries x 4 interleaved groups of partials, combined in group order
  __shared__ float red[4][3][64];
  const int lane = threadIdx.x & 63, grp = threadIdx.x >> 6;
  const int i = blockIdx.x * 64 + lane;              // j*64 + k, grid = 64 blocks
  float dA = 0.f, dWd = 0.f, dBm = 0.f;
#pragma unroll 4
  for (int p = grp; p < nparts; p += 4) {
    const float* q = part + (long long)p * ATT_PARTIAL + i;
    dA += q[0]; dWd += q[64 * 64]; dBm += q[2 * 64 * 64];
  }
  red[grp][0][lane] = dA; red[grp][1][lane] = dWd; red[grp][2][lane] = dBm;
  __syncthreads();
  if (grp == 0) {
    dA = ((red[0][0][lane] + red[1][0][lane]) + red[2][0][lane]) + red[3][0][lane];
    dWd = ((red[0][1][lane] + red[1][1][lane]) + red[2][1][lane]) + red[3][1][lane];
    dBm = ((red[0][2][lane] + red[1][2][lane]) + red[2][2][lane]) + red[3][2][lane];
    const int j = i >> 6, k = i & 63;
    float* row = grads + off.fc1_w + j * 256;
    row[k] = dA; row[64 + k] = dBm; row[128 + k] = dBm - dA; row[192 + k] = dWd;
  }
  if (blockIdx.x == 0 && grp == 1) {
    const int j = lane;
    float w = 0.f, b1 = 0.f;
    for (int p = 0; p < nparts; ++p) {
      w += part[(long long)p * ATT_PARTIAL + 3 * 64 * 64 + j];
      b1 += part[(long long)p * ATT_PARTIAL + 3 * 64 * 64 + 64 + j];
    }
    grads[off.fc2_w + j] = w;
    grads[off.fc1_b + j] = b1;
    if (j == 0) {
      float d = 0.f;
      for (int p = 0; p < nparts; ++p) d += part[(long long)p * ATT_PARTIAL + 3 * 64 * 64 + 128];
      grads[off.fc2_b] = d;
    }
  }
}

// ---------------------------------------------------------------------------------
// launchers
// ---------------------------------------------------------------------------------
static int att_bwd_grid(int B) { return min(B, min(sm_count(), ATT_BWD_CTAS_MAX)); }

int launch_attention_forward(const BatchPtrs& in, const float* P, Workspace& w, int branch, int precision, cudaStream_t s) {
  if (precision == NRM_PRECISION_BF16 || precision == NRM_PRECISION_BF16X3) return launch_attention_forward_tc(in, w, branch, precision, s);
  if (precision != NRM_PRECISION_FP32) { set_error("attention: precision %d not built", precision); return NRM_EUNSUPPORTED; }
  const size_t smem = sizeof(AttSmemFwd);
  // w.scores non-null: the score-exporting instantiations
  void (*k)(const double*, const float*, int, int, int, const float*, float*, float*) =
      w.scores != nullptr ? (branch == 0 ? attention_forward_kernel<0, true> : attention_forward_kernel<1, true>)
                          : (branch == 0 ? attention_forward_kernel<0, false> : attention_forward_kernel<1, false>);
  NRM_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  launch_pdl(k, dim3(w.B), dim3(ATT_THREADS), smem, s, in.xh, (const float*)w.xh, w.B, w.H, w.C, P, w.e, w.scores);
  NRM_LAUNCH_CHECK("attention_forward_kernel");
  return NRM_OK;
}

int launch_attention_backward(const BatchPtrs& in, const float* P, Workspace& w, int branch, int precision, cudaStream_t s) {
  if (precision == NRM_PRECISION_BF16 || precision == NRM_PRECISION_BF16X3) {
    if (use_rowstacked()) {
      // row-stacked kernels: sums over rows (weight gradients, dtp); the label branch exports dhid for its input-gradient kernel
      return launch_attention_backward_rs(w, branch, precision, branch == 0, s);
    }
    return launch_attention_backward_tc(in, P, w, branch, precision, s);
  }
  if (precision != NRM_PRECISION_FP32) { set_error("attention: precision %d not built", precision); return NRM_EUNSUPPORTED; }
  const size_t smem = sizeof(AttSmemBwd);
  const int grid = att_bwd_grid(w.B);
  float* part = w.att_part + (long long)branch * ATT_BWD_CTAS_MAX * ATT_PARTIAL;
  if (branch == 0) {
    NRM_CUDA(cudaFuncSetAttribute(attention_backward_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    launch_pdl(attention_backward_kernel<0>, dim3(grid), dim3(ATT_THREADS), smem, s, in.xh, w.xh, w.B, w.H, w.C, P, w.e, w.de, w.dxh, w.dxt, part);
  } else {
    NRM_CUDA(cudaFuncSetAttribute(attention_backward_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    launch_pdl(attention_backward_kernel<1>, dim3(grid), dim3(ATT_THREADS), smem, s, in.xh, w.xh, w.B, w.H, w.C, P, w.e, w.de, w.dxh, w.dxt, part);
  }
  NRM_LAUNCH_CHECK("attention_backward_kernel");
  return NRM_OK;
}

int launch_attention_finish(const float* P, Workspace& w, int branch, int precision, float* grads, cudaStream_t s) {
  if (precision != NRM_PRECISION_FP32) return branch == 1 ? launch_attention_finish_tc(P, w, grads, s) : NRM_OK;   // one pass for both branches
  const float* part = w.att_part + (long long)branch * ATT_BWD_CTAS_MAX * ATT_PARTIAL;
  launch_pdl(attention_compose_kernel, dim3(64), dim3(256), 0, s, part, att_bwd_grid(w.B), branch == 0 ? ATT_LABEL : ATT_TI, grads);
  NRM_LAUNCH_CHECK("attention_compose_kernel");
  return NRM_OK;
}

}  // namespace nrm
