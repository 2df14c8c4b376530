// Scoring head of UserModel (models/user_model.py:31-35), fused -- the FFMA implementation of precision = fp32 (the other
// precisions run the tensor-core head, nrm_head_tc.cu; head_grad_finish_kernel and the transposes below serve both):
//
//     z = BatchNorm(e);  gate = fc2(gelu(fc1(z)));  x = gate * e;  y = fc2(gelu(fc1(x)));  r = fc2(gelu(fc1(y)))
// Forward: ONE kernel takes a tile of candidate rows through all six layers with the activations in shared
// memory (the five 264 <-> 66 matrices stream through L2, 350 KB per tile); only what the backward needs
// (a1, gate, a2, y, a3) goes back to global memory.
// Backward: kernel A walks the same tile backwards through the data-gradient chain (it reads the nn.Linear
// weights in their natural [out][in] layout: every contraction here has the output index contiguous), writes the
// per-layer gradients of the pre-activations and per-tile partial sums for BatchNorm and out_mlp.fc2; kernel B
// forms the five weight gradients dW = P^T Q over row chunks with 8 x 8 register tiles; a last kernel adds the chunk
// partials in fixed order (deterministic, no atomics).
#include "nrm_kernels.cuh"
#include "nrm_umma.cuh"      // mbarrier helpers

namespace nrm {

constexpr int HT_ROWS = 36;        // candidate rows per tile: 5120 rows (B=1024, C=5) -> 143 tiles, one wave of 148 SMs
constexpr int HT_RPT = 9;          // rows per thread (4 row groups)
constexpr int HT_CONSUMERS = 288;  // 4 x 66 = 264 working threads, 9 warps: the layers
constexpr int HT_THREADS = 320;    // + warp 9: its first lane streams the weight chunks with bulk async copies (TMA engine)
constexpr int LDW = 268;           // row stride of the 264-wide shared buffers (16-byte aligned rows)
constexpr int LDN = 68;            // row stride of the 66-wide shared buffers

constexpr int WCHUNK = 64 * HID;   // floats per staged weight chunk: 64 contraction rows x 66 or 16 x 264
constexpr int W_STAGES = 3;        // ring depth: chunk g is multiplied while g + 1 and g + 2 are in flight
constexpr int W_LAYER_CHUNKS = 5;  // ceil(264 / 64) = ceil(66 / 16) = 5 chunks per layer
constexpr int W_CHUNKS = 5 * W_LAYER_CHUNKS;
struct HeadSmem {
  __align__(16) float w0[HT_ROWS * LDW];
  __align__(16) float w1[HT_ROWS * LDW];   // forward: the e tile; backward: cross row-group reduction scratch [4][2][264]
  __align__(16) float nb[HT_ROWS * LDN];
  __align__(16) float wbuf[W_STAGES][WCHUNK];   // ring of weight chunks (cp.async, two chunks in flight)
  uint64_t full[W_STAGES];               // chunk landed in the slot (complete_tx of the bulk copy)
  uint64_t empty[W_STAGES];              // the nine consumer warps have finished with the slot
};

// Transposed copies of the five matrices for the forward pass: wt = [G1^T | G2^T | M1^T | M2^T | O1^T], each stored
// [contraction index][output index] (output contiguous), same element count as the original.
constexpr int WT_G1 = 0, WT_G2 = HID * E, WT_M1 = 2 * HID * E, WT_M2 = 3 * HID * E, WT_O1 = 4 * HID * E, WT_TOTAL = 5 * HID * E;
static_assert(WT_TOTAL == HEAD_WT_W1T, "w1^T follows the five head matrices in the transposed-weights buffer");

__global__ void __launch_bounds__(256)
head_transpose_kernel(const float* __restrict__ P, float* __restrict__ wt) {
  pdl_wait();                                          // programmatic dependent launch: see nrm_common.cuh
  pdl_trigger();
  const int m = blockIdx.y;                                  // matrix; 5 = w1.weight [64][66] of the history projection
  const long long src_off[6] = {P_GATE_FC1_W, P_GATE_FC2_W, P_MLP_FC1_W, P_MLP_FC2_W, P_OUT_FC1_W, P_W1_W};
  const int rows = m == 5 ? 64 : (m == 1 || m == 3) ? E : HID;             // source is [rows][cols] = [out][in]
  const int cols = m == 5 ? XIN : (m == 1 || m == 3) ? HID : E;
  const float* src = P + src_off[m];
  float* dst = wt + (long long)m * HID * E;                  // [cols][rows]
  for (int i = blockIdx.x * 256 + threadIdx.x; i < rows * cols; i += gridDim.x * 256) {
    const int c = i / rows, r = i - c * rows;                // consecutive threads write consecutive dst elements
    dst[i] = __ldg(src + r * cols + c);
  }
}

// The weights of the five layers a kernel walks through stream through shared memory as ONE sequence of 25 chunks
// (64 x 66 or 16 x 264 floats, 16.9 KB) in a three-slot ring, across layer boundaries, so a layer never starts with a cold
// fetch.  Producer / consumer pipeline: the first lane of warp 9 issues one bulk async copy per chunk
// (cp.async.bulk ... mbarrier::complete_tx: the TMA engine moves the 16.9 KB, no thread touches the data), arming the
// slot's `full` barrier with the byte count; the nine consumer warps wait on `full`, multiply, and arrive on the slot's
// `empty` barrier (one arrival per warp), which the producer waits for before refilling the slot.  No CTA-wide barrier
// per chunk: the consumer warps drift apart by up to the ring depth.
struct HeadLayerDesc { const float* W; int K; int nout; };

// bar.sync is the ALIGNED barrier: a warp must arrive converged (a diverged warp arriving in two groups releases it early)
__device__ __forceinline__ void consumer_sync() { __syncwarp(); asm volatile("bar.sync 1, %0;\n" ::"n"(HT_CONSUMERS) : "memory"); }

__device__ __forceinline__ void weight_producer(HeadSmem& sm, const HeadLayerDesc (&layers)[5]) {
  for (int g = 0; g < W_CHUNKS; ++g) {
    const int l = g / W_LAYER_CHUNKS, c = g - l * W_LAYER_CHUNKS;
    const int kc = WCHUNK / layers[l].nout;
    const int rows = min(kc, layers[l].K - c * kc);
    const float* src = layers[l].W + (long long)c * kc * layers[l].nout;
    const uint32_t bytes = (uint32_t)(rows * layers[l].nout * sizeof(float));
    const int slot = g % W_STAGES, use = g / W_STAGES;
    if (use > 0) umma::mbar_wait(&sm.empty[slot], (uint32_t)((use - 1) & 1));
    const uint32_t bar = umma::smem_u32(&sm.full[slot]);
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(bar), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::"r"(
                     umma::smem_u32(sm.wbuf[slot])), "l"(src), "r"(bytes), "r"(bar) : "memory");
  }
}

// acc[i][q] += sum_k in[(rg*9+i)][k] * W[k][n + 66 q]   (W = [K][66 NQ], output index contiguous), W = layer `layer` of the
// kernel's weight stream.  Called by every CONSUMER thread (threads with work == false only take part in the barriers).
template <int K, int NQ, int LDI>
__device__ __forceinline__ void head_layer(const float* in, HeadSmem& sm, int layer, bool work, int rg, int n, float acc[HT_RPT][NQ]) {
  constexpr int NOUT = HID * NQ;
  constexpr int KC = WCHUNK / NOUT;                      // 64 (NQ = 1) or 16 (NQ = 4)
  constexpr int NCH = (K + KC - 1) / KC;
  static_assert(NCH == W_LAYER_CHUNKS, "chunk table assumes five chunks per layer");
  const float* inr = in + rg * HT_RPT * LDI;
#pragma unroll 1
  for (int c = 0; c < NCH; ++c) {
    const int g = layer * W_LAYER_CHUNKS + c;
    const int slot = g % W_STAGES;
    umma::mbar_wait(&sm.full[slot], (uint32_t)((g / W_STAGES) & 1));      // chunk g has landed
    if (work) {
      const float* wb = sm.wbuf[slot];
      const int kc = (K - c * KC) < KC ? (K - c * KC) : KC;
      const int kc4 = kc & ~3;
      const float* inc = inr + c * KC;
#pragma unroll 4
      for (int k0 = 0; k0 < kc4; k0 += 4) {
        float w[4][NQ];
#pragma unroll
        for (int kk = 0; kk < 4; ++kk)
#pragma unroll
          for (int q = 0; q < NQ; ++q) w[kk][q] = wb[(k0 + kk) * NOUT + n + HID * q];
#pragma unroll
        for (int i = 0; i < HT_RPT; ++i) {
          const float4 a = *reinterpret_cast<const float4*>(inc + i * LDI + k0);
#pragma unroll
          for (int q = 0; q < NQ; ++q) {
            acc[i][q] = fmaf(a.x, w[0][q], acc[i][q]);
            acc[i][q] = fmaf(a.y, w[1][q], acc[i][q]);
            acc[i][q] = fmaf(a.z, w[2][q], acc[i][q]);
            acc[i][q] = fmaf(a.w, w[3][q], acc[i][q]);
          }
        }
      }
      for (int k = kc4; k < kc; ++k) {
        float w[NQ];
#pragma unroll
        for (int q = 0; q < NQ; ++q) w[q] = wb[k * NOUT + n + HID * q];
#pragma unroll
        for (int i = 0; i < HT_RPT; ++i) {
          const float a = inc[i * LDI + k];
#pragma unroll
          for (int q = 0; q < NQ; ++q) acc[i][q] = fmaf(a, w[q], acc[i][q]);
        }
      }
    }
    __syncwarp();
    if ((threadIdx.x & 31) == 0) umma::mbar_arrive(&sm.empty[slot]);       // this warp is done with the slot
  }
}

template <int NQ>
__device__ __forceinline__ void zero_acc(float acc[HT_RPT][NQ]) {
#pragma unroll
  for (int i = 0; i < HT_RPT; ++i)
#pragma unroll
    for (int q = 0; q < NQ; ++q) acc[i][q] = 0.f;
}

// ---------------------------------------------------------------------------------
// forward
// ---------------------------------------------------------------------------------
__global__ void __launch_bounds__(HT_THREADS, 1)
head_forward_kernel(const float* __restrict__ e, const double* __restrict__ bn_sums, long long bn_rows, int training,
                    float* __restrict__ run_mean, float* __restrict__ run_var, long long* __restrict__ nbt,
                    float* __restrict__ mean_out, float* __restrict__ rstd_out,
                    const float* __restrict__ P, const float* __restrict__ wt, long long R, int keep,
                    float* __restrict__ a1g, float* __restrict__ gateg, float* __restrict__ a2g, float* __restrict__ yg,
                    float* __restrict__ a3g, float* __restrict__ logits) {
  pdl_wait();                                          // programmatic dependent launch: see nrm_common.cuh
  pdl_trigger();
  extern __shared__ __align__(16) unsigned char hs_raw[];
  HeadSmem& sm = *reinterpret_cast<HeadSmem*>(hs_raw);
  const int tid = threadIdx.x;
  const long long r0 = (long long)blockIdx.x * HT_ROWS;
  const int nr = (int)min((long long)HT_ROWS, R - r0);
  {
    const HeadLayerDesc layers[5] = {{wt + WT_G1, E, HID}, {wt + WT_G2, HID, E}, {wt + WT_M1, E, HID}, {wt + WT_M2, HID, E}, {wt + WT_O1, E, HID}};
    // barriers of the weight ring, then the roles split: warp 9 streams the weights and leaves
    if (tid == 0) {
      for (int j = 0; j < W_STAGES; ++j) { umma::mbar_init(&sm.full[j], 1); umma::mbar_init(&sm.empty[j], HT_CONSUMERS / 32); }
    }
    __syncthreads();
    if (tid >= HT_CONSUMERS) {
      if (tid == HT_CONSUMERS) weight_producer(sm, layers);
      return;
    }
  }
  // e tile -> w1 (kept for the gating product), z = BatchNorm(e) -> w0.  All loads of the tile are issued first.
  {
    constexpr int NV = HT_ROWS * (E / 4), IT = (NV + HT_CONSUMERS - 1) / HT_CONSUMERS;
    float4 ev[IT];
#pragma unroll
    for (int u = 0; u < IT; ++u) {
      const int i = tid + u * HT_CONSUMERS, r = i / (E / 4), c4 = i - r * (E / 4);
      ev[u] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (i < NV && r < nr) ev[u] = __ldg(reinterpret_cast<const float4*>(e + (r0 + r) * E) + c4);
    }
    // BatchNorm1d statistics (models/user_model.py:18,32), every CTA for itself: training = batch mean / biased variance
    // from the (global) column sums; eval = running statistics.  CTA 0 also publishes them for the backward kernels and
    // updates the running statistics (momentum 0.1, unbiased variance) as nn.BatchNorm1d does.
    float* mean = sm.nb;
    float* rstd = sm.nb + E;
    if (tid < E) {
      const int n = tid;
      float m, v;
      if (training) {
        const double dm = bn_sums[n] / (double)bn_rows;
        double dv = bn_sums[E + n] / (double)bn_rows - dm * dm;
        if (dv < 0.0) dv = 0.0;
        m = (float)dm; v = (float)dv;
        if (blockIdx.x == 0) {
          const double unbiased = bn_rows > 1 ? dv * (double)bn_rows / (double)(bn_rows - 1) : dv;
          run_mean[n] = (1.f - BN_MOMENTUM) * run_mean[n] + BN_MOMENTUM * m;
          run_var[n] = (1.f - BN_MOMENTUM) * run_var[n] + BN_MOMENTUM * (float)unbiased;
          if (n == 0) *nbt += 1;
        }
      } else {
        m = run_mean[n]; v = run_var[n];
      }
      const float rs = 1.0f / sqrtf(v + BN_EPS);
      mean[n] = m; rstd[n] = rs;
      if (blockIdx.x == 0) { mean_out[n] = m; rstd_out[n] = rs; }
    }
    consumer_sync();
#pragma unroll
    for (int u = 0; u < IT; ++u) {
      const int i = tid + u * HT_CONSUMERS, r = i / (E / 4), c4 = i - r * (E / 4);
      if (i >= NV) continue;
      const float4 v = ev[u];
      float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
      if (r < nr) {
        const float4 mu = reinterpret_cast<const float4*>(mean)[c4], rs = reinterpret_cast<const float4*>(rstd)[c4];
        const float4 ga = __ldg(reinterpret_cast<const float4*>(P + P_BN_W) + c4), be = __ldg(reinterpret_cast<const float4*>(P + P_BN_B) + c4);
        z.x = (v.x - mu.x) * rs.x * ga.x + be.x; z.y = (v.y - mu.y) * rs.y * ga.y + be.y;
        z.z = (v.z - mu.z) * rs.z * ga.z + be.z; z.w = (v.w - mu.w) * rs.w * ga.w + be.w;
      }
      *reinterpret_cast<float4*>(sm.w1 + r * LDW + 4 * c4) = v;
      *reinterpret_cast<float4*>(sm.w0 + r * LDW + 4 * c4) = z;
    }
  }
  consumer_sync();
  const bool work = tid < 4 * HID;
  const int rg = work ? tid / HID : 0, n = work ? tid % HID : 0;
  const int rb = rg * HT_RPT;

  // narrow layer: out[r][n] = acc + bias[n]; keep -> global [R][66]; nb = gelu(out)
  auto narrow_out = [&](float acc[HT_RPT][1], const float* bias, float* glob) {
    const float b = __ldg(bias + n);
#pragma unroll
    for (int i = 0; i < HT_RPT; ++i) {
      const float v = acc[i][0] + b;
      if (keep && rb + i < nr) glob[(r0 + rb + i) * HID + n] = v;
      sm.nb[(rb + i) * LDN + n] = gelu_f(v);
    }
  };

  {  // gate.fc1
    float acc[HT_RPT][1]; zero_acc<1>(acc);
    head_layer<E, 1, LDW>(sm.w0, sm, 0, work, rg, n, acc);
    if (work) narrow_out(acc, P + P_GATE_FC1_B, a1g);
  }
  consumer_sync();
  {  // gate.fc2; x = gate * e -> w0
    float acc[HT_RPT][4]; zero_acc<4>(acc);
    head_layer<HID, 4, LDN>(sm.nb, sm, 1, work, rg, n, acc);
    if (work) {
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int k = n + HID * q;
        const float b = __ldg(P + P_GATE_FC2_B + k);
#pragma unroll
        for (int i = 0; i < HT_RPT; ++i) {
          const float g = acc[i][q] + b;
          if (keep && rb + i < nr) gateg[(r0 + rb + i) * E + k] = g;
          sm.w0[(rb + i) * LDW + k] = g * sm.w1[(rb + i) * LDW + k];
        }
      }
    }
  }
  consumer_sync();
  {  // mlp.fc1
    float acc[HT_RPT][1]; zero_acc<1>(acc);
    head_layer<E, 1, LDW>(sm.w0, sm, 2, work, rg, n, acc);
    if (work) narrow_out(acc, P + P_MLP_FC1_B, a2g);
  }
  consumer_sync();
  {  // mlp.fc2 -> y -> w0
    float acc[HT_RPT][4]; zero_acc<4>(acc);
    head_layer<HID, 4, LDN>(sm.nb, sm, 3, work, rg, n, acc);
    if (work) {
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int k = n + HID * q;
        const float b = __ldg(P + P_MLP_FC2_B + k);
#pragma unroll
        for (int i = 0; i < HT_RPT; ++i) {
          const float v = acc[i][q] + b;
          if (keep && rb + i < nr) yg[(r0 + rb + i) * E + k] = v;
          sm.w0[(rb + i) * LDW + k] = v;
        }
      }
    }
  }
  consumer_sync();
  {  // out_mlp.fc1
    float acc[HT_RPT][1]; zero_acc<1>(acc);
    head_layer<E, 1, LDW>(sm.w0, sm, 4, work, rg, n, acc);
    if (work) narrow_out(acc, P + P_OUT_FC1_B, a3g);
  }
  consumer_sync();
  // out_mlp.fc2: one warp per row
  for (int r = tid >> 5; r < nr; r += HT_CONSUMERS / 32) {
    const int lane = tid & 31;
    float acc = 0.f;
    for (int c = lane; c < HID; c += 32) acc = fmaf(sm.nb[r * LDN + c], __ldg(P + P_OUT_FC2_W + c), acc);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) logits[r0 + r] = acc + __ldg(P + P_OUT_FC2_B);
  }
}

// ---------------------------------------------------------------------------------
// backward A: data-gradient chain per row tile.
// tile partial (floats): dO2[66] | do2 | pad -> 68 ; then doubles: bn sums [2][264]
// ---------------------------------------------------------------------------------
constexpr int HB_F = 68;

__global__ void __launch_bounds__(HT_THREADS, 1)
head_backward_kernel(const float* __restrict__ e, const float* __restrict__ mean, const float* __restrict__ rstd,
                     const float* __restrict__ P, long long R, const float* __restrict__ dr,
                     const float* __restrict__ a1g, const float* __restrict__ gateg, const float* __restrict__ a2g,
                     const float* __restrict__ a3g,
                     float* __restrict__ da3g, float* __restrict__ dyg, float* __restrict__ da2g, float* __restrict__ dgateg,
                     float* __restrict__ da1g, float* __restrict__ dzg, float* __restrict__ deg,
                     float* __restrict__ part_f, double* __restrict__ part_bn) {
  pdl_wait();                                          // programmatic dependent launch: see nrm_common.cuh
  pdl_trigger();
  extern __shared__ __align__(16) unsigned char hs_raw[];
  HeadSmem& sm = *reinterpret_cast<HeadSmem*>(hs_raw);
  const int tid = threadIdx.x;
  const long long r0 = (long long)blockIdx.x * HT_ROWS;
  const int nr = (int)min((long long)HT_ROWS, R - r0);
  const bool work = tid < 4 * HID;
  const int rg = work ? tid / HID : 0, n = work ? tid % HID : 0;
  const int rb = rg * HT_RPT;
  float* red = sm.w1;
  {
    // data-gradient chain: the nn.Linear weights in their natural [out][in] layout (the contraction runs over `out`)
    const HeadLayerDesc layers[5] = {{P + P_OUT_FC1_W, HID, E}, {P + P_MLP_FC2_W, E, HID}, {P + P_MLP_FC1_W, HID, E},
                                     {P + P_GATE_FC2_W, E, HID}, {P + P_GATE_FC1_W, HID, E}};
    // barriers of the weight ring, then the roles split: warp 9 streams the weights and leaves
    if (tid == 0) {
      for (int j = 0; j < W_STAGES; ++j) { umma::mbar_init(&sm.full[j], 1); umma::mbar_init(&sm.empty[j], HT_CONSUMERS / 32); }
    }
    __syncthreads();
    if (tid >= HT_CONSUMERS) {
      if (tid == HT_CONSUMERS) weight_producer(sm, layers);
      return;
    }
  }

  // da3 = dr * O2 * gelu'(a3) -> nb; dO2 / do2 partial sums
  if (work) {
    const float o2 = __ldg(P + P_OUT_FC2_W + n);
    float dw = 0.f, db = 0.f;
#pragma unroll
    for (int i = 0; i < HT_RPT; ++i) {
      float d = 0.f;
      if (rb + i < nr) {
        const float drr = __ldg(dr + r0 + rb + i);
        float gp;
        const float g = gelu_both(__ldg(a3g + (r0 + rb + i) * HID + n), gp);
        d = drr * o2 * gp;
        dw = fmaf(drr, g, dw);
        db += drr;
        da3g[(r0 + rb + i) * HID + n] = d;
      }
      sm.nb[(rb + i) * LDN + n] = d;
    }
    red[rg * 2 * E + n] = dw;
    if (n == 0) red[rg * 2 * E + E] = db;
  }
  consumer_sync();
  if (tid < HID) part_f[(long long)blockIdx.x * HB_F + tid] = ((red[tid] + red[2 * E + tid]) + red[4 * E + tid]) + red[6 * E + tid];
  if (tid == HID) part_f[(long long)blockIdx.x * HB_F + HID] = ((red[E] + red[2 * E + E]) + red[4 * E + E]) + red[6 * E + E];

  {  // dy = da3 O1 -> w0
    float acc[HT_RPT][4]; zero_acc<4>(acc);
    head_layer<HID, 4, LDN>(sm.nb, sm, 0, work, rg, n, acc);
    if (work) {
#pragma unroll
      for (int q = 0; q < 4; ++q)
#pragma unroll
        for (int i = 0; i < HT_RPT; ++i) {
          const int k = n + HID * q;
          if (rb + i < nr) dyg[(r0 + rb + i) * E + k] = acc[i][q];
          sm.w0[(rb + i) * LDW + k] = acc[i][q];
        }
    }
  }
  consumer_sync();
  {  // da2 = (dy M2) * gelu'(a2) -> nb
    float acc[HT_RPT][1]; zero_acc<1>(acc);
    head_layer<E, 1, LDW>(sm.w0, sm, 1, work, rg, n, acc);
    if (work) {
#pragma unroll
      for (int i = 0; i < HT_RPT; ++i) {
        float d = 0.f;
        if (rb + i < nr) {
          d = acc[i][0] * gelu_grad_f(__ldg(a2g + (r0 + rb + i) * HID + n));
          da2g[(r0 + rb + i) * HID + n] = d;
        }
        sm.nb[(rb + i) * LDN + n] = d;
      }
    }
  }
  consumer_sync();
  {  // dx = da2 M1;  dgate = dx * e -> w0;  de (direct path) = dx * gate
    float acc[HT_RPT][4]; zero_acc<4>(acc);
    head_layer<HID, 4, LDN>(sm.nb, sm, 2, work, rg, n, acc);
    if (work) {
#pragma unroll
      for (int q = 0; q < 4; ++q)
#pragma unroll
        for (int i = 0; i < HT_RPT; ++i) {
          const int k = n + HID * q;
          float dg = 0.f;
          if (rb + i < nr) {
            const long long gi = (r0 + rb + i) * E + k;
            dg = acc[i][q] * __ldg(e + gi);
            dgateg[gi] = dg;
            deg[gi] = acc[i][q] * __ldg(gateg + gi);
          }
          sm.w0[(rb + i) * LDW + k] = dg;
        }
    }
  }
  consumer_sync();
  {  // da1 = (dgate G2) * gelu'(a1) -> nb
    float acc[HT_RPT][1]; zero_acc<1>(acc);
    head_layer<E, 1, LDW>(sm.w0, sm, 3, work, rg, n, acc);
    if (work) {
#pragma unroll
      for (int i = 0; i < HT_RPT; ++i) {
        float d = 0.f;
        if (rb + i < nr) {
          d = acc[i][0] * gelu_grad_f(__ldg(a1g + (r0 + rb + i) * HID + n));
          da1g[(r0 + rb + i) * HID + n] = d;
        }
        sm.nb[(rb + i) * LDN + n] = d;
      }
    }
  }
  consumer_sync();
  {  // dz = da1 G1; BatchNorm partial sums of dz and dz * xhat over this tile's rows
    float acc[HT_RPT][4]; zero_acc<4>(acc);
    head_layer<HID, 4, LDN>(sm.nb, sm, 4, work, rg, n, acc);
    if (work) {
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int k = n + HID * q;
        const float mu = __ldg(mean + k), rs = __ldg(rstd + k);
        float s = 0.f, sx = 0.f;
#pragma unroll
        for (int i = 0; i < HT_RPT; ++i) {
          if (rb + i < nr) {
            const long long gi = (r0 + rb + i) * E + k;
            const float d = acc[i][q];
            dzg[gi] = d;
            s += d;
            sx = fmaf(d, (__ldg(e + gi) - mu) * rs, sx);
          }
        }
        red[rg * 2 * E + k] = s;
        red[rg * 2 * E + E + k] = sx;
      }
    }
  }
  consumer_sync();
  for (int i = tid; i < 2 * E; i += HT_CONSUMERS)
    part_bn[(long long)blockIdx.x * 2 * E + i] = ((double)red[i] + (double)red[2 * E + i]) + ((double)red[4 * E + i] + (double)red[6 * E + i]);
}

// ---------------------------------------------------------------------------------
// backward B: weight gradients.  blockIdx.y = layer, blockIdx.x = row chunk.
//   dW[nn][kk] = sum_r Pm[r][nn] * Q[r][kk],  nn < 66 (narrow side), kk < 264 (wide side); thread kk keeps 66 sums.
//   layer 0 out_mlp.fc1: Pm = da3,        Q = y          bias = colsum(Pm)        weight is [66][264]
//   layer 1 mlp.fc2    : Pm = gelu(a2),   Q = dy         bias = colsum(Q)         weight is [264][66]
//   layer 2 mlp.fc1    : Pm = da2,        Q = gate * e   bias = colsum(Pm)
//   layer 3 gate.fc2   : Pm = gelu(a1),   Q = dgate      bias = colsum(Q)
//   layer 4 gate.fc1   : Pm = da1,        Q = BN(e)      bias = colsum(Pm)
// chunk partial (floats): [66][264] in (nn, kk) order | bias[264 (padded)]
// ---------------------------------------------------------------------------------
constexpr int WG_THREADS = 320, WG_TILE = 32, WG_PART = HID * E + E;
constexpr int WG_LDP = 72;          // row stride of the narrow-side tile (66 padded to 9 groups of 8)

// thread (ng, kg) owns the 8 x 8 block dW[8 ng .. +8][{4 kg .. +4} u {132 + 4 kg .. +4}] (two 4-wide column groups, so
// that the lanes of a warp read consecutive 16-byte words of the wide tile): per row two 16-byte reads of each operand feed 64 FMAs
__global__ void __launch_bounds__(WG_THREADS, 1)
head_wgrad_kernel(const float* __restrict__ e, const float* __restrict__ mean, const float* __restrict__ rstd,
                  const float* __restrict__ P, long long R, int rows_per_chunk,
                  const float* __restrict__ a1g, const float* __restrict__ gateg, const float* __restrict__ a2g,
                  const float* __restrict__ yg, const float* __restrict__ da3g, const float* __restrict__ dyg,
                  const float* __restrict__ da2g, const float* __restrict__ dgateg, const float* __restrict__ da1g,
                  float* __restrict__ part) {
  pdl_wait();                                          // programmatic dependent launch: see nrm_common.cuh
  pdl_trigger();
  __shared__ __align__(16) float sp[WG_TILE][WG_LDP];
  __shared__ __align__(16) float sq[WG_TILE][E];
  const int layer = blockIdx.y, tid = threadIdx.x;
  const long long rbeg = (long long)blockIdx.x * rows_per_chunk;
  const long long rend = min(R, rbeg + rows_per_chunk);
  const float* Psrc = layer == 0 ? da3g : layer == 1 ? a2g : layer == 2 ? da2g : layer == 3 ? a1g : da1g;
  const float* Qsrc = layer == 0 ? yg : layer == 1 ? dyg : layer == 2 ? gateg : layer == 3 ? dgateg : e;
  const bool p_gelu = (layer == 1 || layer == 3);
  const bool wide_bias = (layer == 1 || layer == 3);
  const bool work = tid < 9 * 33;
  const int ng = work ? tid / 33 : 0, kg = work ? tid % 33 : 0;
  float acc[8][8];
#pragma unroll
  for (int a = 0; a < 8; ++a)
#pragma unroll
    for (int b = 0; b < 8; ++b) acc[a][b] = 0.f;
  float bsum[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  for (int i = tid; i < WG_TILE * (WG_LDP - HID); i += WG_THREADS) sp[i / (WG_LDP - HID)][HID + i % (WG_LDP - HID)] = 0.f;   // pad columns
  for (long long t0 = rbeg; t0 < rend; t0 += WG_TILE) {
    const int nt = (int)min((long long)WG_TILE, rend - t0);
    __syncthreads();
    {
      // all global loads of the two tiles first (independent requests in flight), then the transforms and stores
      constexpr int NPV = WG_TILE * HID, ITP = (NPV + WG_THREADS - 1) / WG_THREADS;
      constexpr int NQV = WG_TILE * (E / 4), ITQ = (NQV + WG_THREADS - 1) / WG_THREADS;
      float pv[ITP];
      float4 qv[ITQ], ev[ITQ];
#pragma unroll
      for (int u = 0; u < ITP; ++u) {
        const int i = tid + u * WG_THREADS, r = i / HID, c = i - r * HID;
        pv[u] = (i < NPV && r < nt) ? __ldg(Psrc + (t0 + r) * HID + c) : 0.f;
      }
#pragma unroll
      for (int u = 0; u < ITQ; ++u) {
        const int i = tid + u * WG_THREADS, r = i / (E / 4), c4 = i - r * (E / 4);
        const bool ok = i < NQV && r < nt;
        qv[u] = ok ? __ldg(reinterpret_cast<const float4*>(Qsrc + (t0 + r) * E) + c4) : make_float4(0.f, 0.f, 0.f, 0.f);
        if (layer == 2) ev[u] = ok ? __ldg(reinterpret_cast<const float4*>(e + (t0 + r) * E) + c4) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
#pragma unroll
      for (int u = 0; u < ITP; ++u) {
        const int i = tid + u * WG_THREADS, r = i / HID, c = i - r * HID;
        if (i < NPV) sp[r][c] = (p_gelu && r < nt) ? gelu_f(pv[u]) : pv[u];
      }
#pragma unroll
      for (int u = 0; u < ITQ; ++u) {
        const int i = tid + u * WG_THREADS, r = i / (E / 4), c4 = i - r * (E / 4);
        if (i >= NQV) continue;
        float4 q = qv[u];
        if (r < nt) {
          if (layer == 2) {
            q.x *= ev[u].x; q.y *= ev[u].y; q.z *= ev[u].z; q.w *= ev[u].w;
          } else if (layer == 4) {
            const float4 mu = __ldg(reinterpret_cast<const float4*>(mean) + c4), rs = __ldg(reinterpret_cast<const float4*>(rstd) + c4);
            const float4 ga = __ldg(reinterpret_cast<const float4*>(P + P_BN_W) + c4), be = __ldg(reinterpret_cast<const float4*>(P + P_BN_B) + c4);
            q.x = (q.x - mu.x) * rs.x * ga.x + be.x; q.y = (q.y - mu.y) * rs.y * ga.y + be.y;
            q.z = (q.z - mu.z) * rs.z * ga.z + be.z; q.w = (q.w - mu.w) * rs.w * ga.w + be.w;
          }
        }
        *reinterpret_cast<float4*>(&sq[r][4 * c4]) = q;
      }
    }
    __syncthreads();
    if (work) {
#pragma unroll 4
      for (int r = 0; r < WG_TILE; ++r) {
        const float4 p0 = *reinterpret_cast<const float4*>(&sp[r][8 * ng]), p1 = *reinterpret_cast<const float4*>(&sp[r][8 * ng + 4]);
        const float4 q0 = *reinterpret_cast<const float4*>(&sq[r][4 * kg]), q1 = *reinterpret_cast<const float4*>(&sq[r][E / 2 + 4 * kg]);
        const float pv[8] = {p0.x, p0.y, p0.z, p0.w, p1.x, p1.y, p1.z, p1.w};
        const float qv[8] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w};
#pragma unroll
        for (int a = 0; a < 8; ++a)
#pragma unroll
          for (int b = 0; b < 8; ++b) acc[a][b] = fmaf(pv[a], qv[b], acc[a][b]);
        if (wide_bias) {
#pragma unroll
          for (int b = 0; b < 8; ++b) bsum[b] += qv[b];
        } else {
#pragma unroll
          for (int a = 0; a < 8; ++a) bsum[a] += pv[a];
        }
      }
    }
  }
  float* out = part + ((long long)layer * gridDim.x + blockIdx.x) * WG_PART;
  if (work) {
#pragma unroll
    for (int a = 0; a < 8; ++a) {
      const int nn = 8 * ng + a;
      if (nn < HID) {
        *reinterpret_cast<float4*>(out + nn * E + 4 * kg) = make_float4(acc[a][0], acc[a][1], acc[a][2], acc[a][3]);
        *reinterpret_cast<float4*>(out + nn * E + E / 2 + 4 * kg) = make_float4(acc[a][4], acc[a][5], acc[a][6], acc[a][7]);
      }
    }
    if (wide_bias) {
      if (ng == 0) {
#pragma unroll
        for (int b = 0; b < 8; ++b) out[HID * E + (b < 4 ? 4 * kg + b : E / 2 + 4 * kg + b - 4)] = bsum[b];
      }
    } else if (kg == 0) {
#pragma unroll
      for (int a = 0; a < 8; ++a) if (8 * ng + a < HID) out[HID * E + 8 * ng + a] = bsum[a];
    }
  }
}

// Sum the chunk partials and write the head gradients (transposing layers 1 and 3, whose weights are [264][66]); also
// out_mlp.fc2 from the tile partials of kernel A and the BatchNorm sums.  Block = 64 consecutive entries x 4 interleaved
// groups of partials (group g adds partials g, g + 4, ... in order; the four group sums are combined in group order):
// fixed summation order, chains a quarter as long.
constexpr int GF_ENT = 64;
__global__ void __launch_bounds__(256)
head_grad_finish_kernel(const float* __restrict__ part, int nchunks, const float* __restrict__ part_f, int ntiles,
                        const double* __restrict__ part_bn, float* __restrict__ grads, double* __restrict__ bn_bwd_sums, int layer_base) {
  pdl_wait();                                          // programmatic dependent launch: see nrm_common.cuh
  pdl_trigger();
  __shared__ double red[4][GF_ENT];
  const int layer = layer_base + blockIdx.y;           // 0-4 weight gradients, 5 out_mlp.fc2, 6 BatchNorm sums
  const int lane = threadIdx.x & (GF_ENT - 1), grp = threadIdx.x >> 6;
  const int i = blockIdx.x * GF_ENT + lane;
  const int nent = layer < 5 ? WG_PART : layer == 5 ? HID + 1 : 2 * E;
  if (blockIdx.x * GF_ENT >= nent) return;
  double s = 0.0;
  if (i < nent) {
    if (layer < 5) {
      const float* src = part + (long long)layer * nchunks * WG_PART + i;
      float f = 0.f;
#pragma unroll 4
      for (int c = grp; c < nchunks; c += 4) f += src[(long long)c * WG_PART];
      s = (double)f;
    } else if (layer == 5) {
      float f = 0.f;
#pragma unroll 4
      for (int t = grp; t < ntiles; t += 4) f += part_f[(long long)t * HB_F + i];
      s = (double)f;
    } else {
#pragma unroll 4
      for (int t = grp; t < ntiles; t += 4) s += part_bn[(long long)t * 2 * E + i];
    }
  }
  red[grp][lane] = s;
  __syncthreads();
  if (grp != 0 || i >= nent) return;
  if (layer < 6) {
    const float v = (((float)red[0][lane] + (float)red[1][lane]) + (float)red[2][lane]) + (float)red[3][lane];
    if (layer < 5) {
      const long long w_off[5] = {P_OUT_FC1_W, P_MLP_FC2_W, P_MLP_FC1_W, P_GATE_FC2_W, P_GATE_FC1_W};
      const long long b_off[5] = {P_OUT_FC1_B, P_MLP_FC2_B, P_MLP_FC1_B, P_GATE_FC2_B, P_GATE_FC1_B};
      if (i < HID * E) {
        const int nn = i / E, kq = i - nn * E;
        if (layer == 1 || layer == 3) grads[w_off[layer] + (long long)kq * HID + nn] = v;
        else grads[w_off[layer] + (long long)nn * E + kq] = v;
      } else {
        const int bi = i - HID * E;
        const int nb = (layer == 1 || layer == 3) ? E : HID;
        if (bi < nb) grads[b_off[layer] + bi] = v;
      }
    } else {
      if (i < HID) grads[P_OUT_FC2_W + i] = v; else grads[P_OUT_FC2_B] = v;
    }
  } else {
    // BatchNorm: column sums of dz and dz * xhat (this rank's rows), bn.weight / bn.bias gradients
    const double v = ((red[0][lane] + red[1][lane]) + red[2][lane]) + red[3][lane];
    bn_bwd_sums[i] = v;
    if (i < E) grads[P_BN_B + i] = (float)v; else grads[P_BN_W + (i - E)] = (float)v;
  }
}

// ---------------------------------------------------------------------------------
// launchers
// ---------------------------------------------------------------------------------
static inline int head_tiles(long long R) { return (int)((R + HT_ROWS - 1) / HT_ROWS); }
int head_wgrad_chunks(long long R) {
  // about two waves of 5-layer CTAs, at least one 32-row tile per chunk
  int n = (2 * sm_count() + 4) / 5;
  const int maxn = (int)((R + WG_TILE - 1) / WG_TILE);
  if (n > maxn) n = maxn;
  if (n > HEAD_WG_CHUNKS_MAX) n = HEAD_WG_CHUNKS_MAX;
  return n < 1 ? 1 : n;
}

// transposed copies of the five matrices for the forward kernel: weights only, enqueued ahead of the encoder
int launch_head_transpose(const float* P, Workspace& w, cudaStream_t s) {
  launch_pdl(head_transpose_kernel, dim3(dim3(8, 6)), dim3(256), 0, s, P, w.head_wt);
  NRM_LAUNCH_CHECK("head_transpose_kernel");
  return NRM_OK;
}

int launch_head_forward_fused(const float* P, Workspace& w, float* run_mean, float* run_var, long long* nbt, int training, int keep,
                              const double* bn_sums, long long bn_rows, float* logits, cudaStream_t s) {
  static DeviceOnce configured;                          // function attributes are per device
  if (configured.first_time()) {
    NRM_CUDA(cudaFuncSetAttribute(head_forward_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(HeadSmem)));
    NRM_CUDA(cudaFuncSetAttribute(head_backward_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(HeadSmem)));
  }
  launch_pdl(head_forward_kernel, dim3(head_tiles(w.R)), dim3(HT_THREADS), sizeof(HeadSmem), s, w.e, bn_sums, bn_rows, training, run_mean, run_var, nbt, w.mean, w.rstd, P, w.head_wt, w.R, keep, w.a1, w.gate, w.a2, w.y, w.a3, logits);
  NRM_LAUNCH_CHECK("head_forward_kernel");
  return NRM_OK;
}

// The head backward in three parts, so that a caller may run the weight gradients beside what follows:
//   dgrad : the data-gradient chain (-> da*, dy, dgate, dz, de and the per-tile partials)
//   bn    : BatchNorm sums from the tile partials (-> w.bn_bwd_sums, bn.weight / bn.bias gradients): needed by the encoder backward
//   wgrad : the five weight gradients + out_mlp.fc2 (only the optimizer needs them)
static void head_wgrad_shape(const Workspace& w, int& rpc, int& nchunks) {
  const int nch = head_wgrad_chunks(w.R);
  rpc = (int)((w.R + nch - 1) / nch);
  rpc = (rpc + WG_TILE - 1) / WG_TILE * WG_TILE;
  nchunks = (int)((w.R + rpc - 1) / rpc);
}

int launch_head_backward_dgrad(const float* P, Workspace& w, const float* dlogits, cudaStream_t s) {
  static DeviceOnce configured;                          // function attributes are per device
  if (configured.first_time()) {
    NRM_CUDA(cudaFuncSetAttribute(head_backward_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(HeadSmem)));
  }
  launch_pdl(head_backward_kernel, dim3(head_tiles(w.R)), dim3(HT_THREADS), sizeof(HeadSmem), s, w.e, w.mean, w.rstd, P, w.R, dlogits, w.a1, w.gate, w.a2, w.a3, w.da3, w.dy, w.da2, w.dgate, w.da1, w.dz, w.de, w.head_part_f, w.head_part_bn);
  NRM_LAUNCH_CHECK("head_backward_kernel");
  return NRM_OK;
}

int launch_head_backward_bn(Workspace& w, float* G, cudaStream_t s, int dgrad_tiles) {
  int rpc, nchunks;
  head_wgrad_shape(w, rpc, nchunks);
  const int ntiles = dgrad_tiles > 0 ? dgrad_tiles : head_tiles(w.R);      // row tiles of the data-gradient kernel that wrote the partials
  launch_pdl(head_grad_finish_kernel, dim3((2 * E + GF_ENT - 1) / GF_ENT, 1), dim3(256), 0, s, w.head_part_w, nchunks, w.head_part_f, ntiles, w.head_part_bn, G, w.bn_bwd_sums, 6);
  NRM_LAUNCH_CHECK("head_grad_finish_kernel");
  return NRM_OK;
}

int launch_head_backward_wgrad(const float* P, Workspace& w, float* G, cudaStream_t s, int dgrad_tiles, int tc_precision) {
  int rpc, nchunks;
  head_wgrad_shape(w, rpc, nchunks);
  const int ntiles = dgrad_tiles > 0 ? dgrad_tiles : head_tiles(w.R);
  if (tc_precision != 0) {
    // tensor-core products: chunks of whole 64-row tiles, about one wave of 5-layer CTAs
    int nch = (sm_count() + 4) / 5;
    const int maxn = (int)((w.R + 63) / 64);
    if (nch > maxn) nch = maxn;
    if (nch > HEAD_WG_CHUNKS_MAX) nch = HEAD_WG_CHUNKS_MAX;
    rpc = (int)(((w.R + nch - 1) / nch + 63) / 64 * 64);
    nchunks = (int)((w.R + rpc - 1) / rpc);
    NRM_TRY(launch_head_wgrad_tc(P, w, tc_precision, rpc, nchunks, s));
  } else
  launch_pdl(head_wgrad_kernel, dim3(nchunks, 5), dim3(WG_THREADS), 0, s, w.e, w.mean, w.rstd, P, w.R, rpc, w.a1, w.gate, w.a2, w.y, w.da3, w.dy, w.da2, w.dgate, w.da1, w.head_part_w);
  NRM_LAUNCH_CHECK("head_wgrad_kernel");
  launch_pdl(head_grad_finish_kernel, dim3((WG_PART + GF_ENT - 1) / GF_ENT, 6), dim3(256), 0, s, w.head_part_w, nchunks, w.head_part_f, ntiles, w.head_part_bn, G, w.bn_bwd_sums, 0);
  NRM_LAUNCH_CHECK("head_grad_finish_kernel");
  return NRM_OK;
}

}  // namespace nrm
