// Backward of w1 = nn.Linear(66, 64) over the embedded history rows (models/user_invariant_interest_model.py:33,78) on the tensor cores.
//   dxin[r][k] = sum_j dxh[r][j] W1[j][k]                                                     M = rows, N = 80, K = 64
//   dW1[j][k]  = sum_r dxh[r][j] xin[r][k],   db1[j] = sum_r dxh[r][j]                        M = 64,  N = 80, K = rows
// NH = B*H rows (51 200 at B = 1024, H = 50; 1 048 576 at B = 4096, H = 256): tall-skinny products whose FFMA versions
// (nrm_w1.cu) spend 25 / 120 us on 0.4 / 0.9 GFLOP.  Here a CTA walks tiles of 128 rows: its threads turn the fp32 rows into
// un-swizzled K-major bf16 operand tiles (hi | lo parts, 3 MMAs per product = fp32-grade, as in the attention kernels) and one
// elected thread issues tcgen05.mma; the weight-gradient product reads the SAME two tiles MN-major (contraction over the rows) and
// accumulates in tensor memory over all tiles of the CTA; db1 rides along as the product with a column of ones (K padding of xin).
// Per-CTA partials are summed in CTA order by w1_finish_kernel (deterministic).  Used when precision != fp32; the forward is
// nrm_w1.cu's FFMA kernel in every precision.
#include "nrm_kernels.cuh"

#include "nrm_umma.cuh"

namespace nrm {
namespace w1tc {

constexpr int ROWS = 128;
constexpr int KX = 80;                        // xin columns padded to a multiple of 16 (66 real, column 66 = 1 in the backward, rest 0)
constexpr uint32_t LBO = ROWS * 16;           // K-major tile of 128 rows: (r, 8 kb) at kb * 2048 + (r / 8) * 128 + (r % 8) * 16
constexpr uint32_t X_TILE = (KX / 8) * LBO;   // 20480 B per part
constexpr uint32_t D_TILE = 8 * LBO;          // 16384 B per part (64 columns)
constexpr int W1_PART = 64 * XIN + 64;        // dW1 [64][66] | db1 [64]  (same partial layout as nrm_w1.cu)

__device__ __forceinline__ uint32_t tile_off(int r, int kb) { return (uint32_t)kb * LBO + (uint32_t)(r >> 3) * 128u + (uint32_t)(r & 7) * 16u; }
// operand views of a 128-row K-major tile with `part` bytes between its hi and lo parts
__device__ __forceinline__ umma::Operand op_k(uint32_t addr, uint32_t part) { return umma::make_operand(addr, LBO, 128, 2 * LBO, part); }
__device__ __forceinline__ umma::Operand op_mn(uint32_t addr, uint32_t part) { return umma::make_operand(addr, 128, LBO, 256, part); }

// W1^T as a K-major tile [80 rows k][64 j] (LBO = 80 rows * 16 B = 1280): B operand of the dxin product
template <int NP>
__device__ __forceinline__ void build_w_kj(const float* __restrict__ W, unsigned char* tile, uint32_t part) {
  for (int it = threadIdx.x; it < KX * 8; it += (int)blockDim.x) {
    const int k = it % KX, jb = it / KX;
    float v[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = (k < XIN) ? __ldg(W + (jb * 8 + i) * XIN + k) : 0.f;
    umma::store_operand8<NP>(tile, (uint32_t)jb * 1280u + (uint32_t)(k >> 3) * 128u + (uint32_t)(k & 7) * 16u, part, v);
  }
}

// fp32 rows already staged in shared memory (row-major, `cols` floats per row, cp.async) -> K-major bf16 tile(s)
template <int NP, int KB>
__device__ __forceinline__ void convert_staged(const float* __restrict__ stg, int cols, int nr, unsigned char* tile, uint32_t part, int one_col) {
  for (int it = threadIdx.x; it < ROWS * KB; it += (int)blockDim.x) {
    const int r = it & (ROWS - 1), kb = it >> 7;
    float v[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = 0.f;
    if (r < nr) {
      const float* p = stg + r * cols + kb * 8;
      if (kb * 8 + 8 <= cols) {
#pragma unroll
        for (int i = 0; i < 4; ++i) { const float2 x = *reinterpret_cast<const float2*>(p + 2 * i); v[2 * i] = x.x; v[2 * i + 1] = x.y; }
      } else {
#pragma unroll
        for (int i = 0; i < 8; ++i) if (kb * 8 + i < cols) v[i] = p[i];
      }
      if (one_col >= 0 && (one_col >> 3) == kb) v[one_col & 7] = 1.0f;
    }
    umma::store_operand8<NP>(tile, tile_off(r, kb), part, v);
  }
}
// a tile of rows is one contiguous block of global memory: 16-byte cp.async, every request in flight at once
__device__ __forceinline__ void stage_rows(float* stg, const float* __restrict__ src, int nfloats) {
  const int n4 = nfloats >> 2;                            // tile starts are multiples of 128 rows: 16-byte aligned; nfloats is even
  for (int i = threadIdx.x; i < n4; i += (int)blockDim.x)
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(umma::smem_u32(stg + 4 * i)), "l"(src + 4 * i) : "memory");
  for (int i = (n4 << 2) + threadIdx.x; i < nfloats; i += (int)blockDim.x) stg[i] = __ldg(src + i);
}

template <int NP>
struct SmemBwd {
  __align__(16) float stg_d[ROWS * 64];                 // fp32 staging of the NEXT tile (cp.async), filled while the products of the current one run
  __align__(16) float stg_x[ROWS * XIN];
  __align__(128) unsigned char ds[NP * D_TILE];         // dxh tile  [128 r][64 j]
  __align__(128) unsigned char xs[NP * X_TILE];         // xin tile  [128 r][80 k], column 66 = 1
  __align__(128) unsigned char wt[NP * KX * 64 * 2];    // W1^T      [80 k][64 j]
  uint64_t mbar;
  uint32_t tmem_base;
};
constexpr uint32_t COL_DX = 0, COL_DW = 128, BWD_COLS = 256;   // dxin accumulator [128][80]; dW1^T-side accumulator [64 j][80 k]

constexpr int BWD_THREADS = 512;              // 16 warps stage and convert the tiles; warps 0-7 read the accumulators back
template <int SPLIT>
__global__ void __launch_bounds__(BWD_THREADS)
w1_backward_tc_kernel(const float* __restrict__ xin, const float* __restrict__ dxh, const float* __restrict__ P, float* __restrict__ dxin,
                      long long NH, float* __restrict__ part) {
  pdl_wait();
  pdl_trigger();
  constexpr int NP = SPLIT == 3 ? 2 : 1;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  SmemBwd<NP>& sm = *reinterpret_cast<SmemBwd<NP>*>(smem_raw);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (tid == 0) umma::mbar_init(&sm.mbar, 1);
  if (warp == 0) umma::tmem_alloc(&sm.tmem_base, BWD_COLS);
  build_w_kj<NP>(P + P_W1_W, sm.wt, KX * 64 * 2);
  umma::fence_async_smem();
  umma::fence_before_sync();
  __syncthreads();
  umma::fence_after_sync();
  const uint32_t tmem = sm.tmem_base;
  constexpr uint32_t IDESC_DX = umma::make_idesc_bf16(128, KX);                // dxh (K-major) x W1^T (K-major)
  constexpr uint32_t IDESC_DW = umma::make_idesc_bf16(64, KX, true, true);     // dxh^T x xin^T: both tiles read MN-major
  const int sp = warp & 3, half = warp >> 2;
  uint32_t phase = 0;
  bool started = false;
  const long long ntiles = (NH + ROWS - 1) / ROWS;
  if ((long long)blockIdx.x < ntiles) {
    const long long r0 = (long long)blockIdx.x * ROWS;
    const int nr = (int)min((long long)ROWS, NH - r0);
    stage_rows(sm.stg_d, dxh + r0 * 64, nr * 64);
    stage_rows(sm.stg_x, xin + r0 * XIN, nr * XIN);
  }
  for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const long long r0 = tile * ROWS;
    const int nr = (int)min((long long)ROWS, NH - r0);
    asm volatile("cp.async.wait_all;\n" ::: "memory");
    __syncthreads();                                   // staged rows visible; the previous tile's products have completed (waited below)
    convert_staged<NP, 8>(sm.stg_d, 64, nr, sm.ds, D_TILE, -1);
    convert_staged<NP, KX / 8>(sm.stg_x, XIN, nr, sm.xs, X_TILE, XIN);         // column 66 := 1 -> db1 comes out of the weight product
    umma::fence_async_smem();
    umma::fence_before_sync();
    __syncthreads();
    {                                                  // the next tile travels while this one is multiplied and written out
      const long long nt = tile + gridDim.x;
      if (nt < ntiles) {
        const int nnr = (int)min((long long)ROWS, NH - nt * ROWS);
        stage_rows(sm.stg_d, dxh + nt * ROWS * 64, nnr * 64);
        stage_rows(sm.stg_x, xin + nt * ROWS * XIN, nnr * XIN);
      }
    }
    if (warp == 0 && umma::elect_one()) {
      umma::fence_after_sync();
      umma::mma_product<SPLIT, 4>(tmem + COL_DX, op_k(umma::smem_u32(sm.ds), D_TILE),
                                  umma::make_operand(umma::smem_u32(sm.wt), 1280, 128, 2560, KX * 64 * 2), IDESC_DX, false);
      umma::mma_product<SPLIT, 8>(tmem + COL_DW, op_mn(umma::smem_u32(sm.ds), D_TILE), op_mn(umma::smem_u32(sm.xs), X_TILE), IDESC_DW, started);
      umma::mma_commit(&sm.mbar);
    }
    started = true;
    umma::mbar_wait(&sm.mbar, phase);
    phase ^= 1;
    umma::fence_after_sync();
    // dxin rows: thread = (row, column half of 40)
    if (warp < 8) {
    float v[40];
    umma::tmem_ld32(tmem + COL_DX + 40 * half + ((uint32_t)(32 * sp) << 16), v);
    umma::tmem_ld8(tmem + COL_DX + 40 * half + 32 + ((uint32_t)(32 * sp) << 16), v + 32);
    umma::fence_before_sync();
    const int r = 32 * sp + lane;
    if (r < nr) {
      float2* dst = reinterpret_cast<float2*>(dxin + (r0 + r) * XIN + 40 * half);
      const int ncol = half == 0 ? 40 : XIN - 40;       // 40 | 26 real columns
#pragma unroll
      for (int q = 0; q < 20; ++q)
        if (2 * q < ncol) dst[q] = make_float2(v[2 * q], v[2 * q + 1]);
    }
    }
  }
  // per-CTA partial of dW1 / db1: an M = 64 accumulator occupies lanes 0-15 of every sub-partition (j = 16 sp + lane)
  umma::fence_after_sync();
  float* out = part + (long long)blockIdx.x * W1_PART;
  if (warp < 8) {
    float v[40];
    umma::tmem_ld32(tmem + COL_DW + 40 * half + ((uint32_t)(32 * sp) << 16), v);
    umma::tmem_ld8(tmem + COL_DW + 40 * half + 32 + ((uint32_t)(32 * sp) << 16), v + 32);
    if (lane < 16) {
      const int j = 16 * sp + lane;
#pragma unroll
      for (int q = 0; q < 40; ++q) {
        const int k = 40 * half + q;
        const float x = started ? v[q] : 0.f;
        if (k < XIN) out[j * XIN + k] = x;
        else if (k == XIN) out[64 * XIN + j] = x;
      }
    }
  }
  umma::fence_before_sync();
  __syncthreads();
  if (warp == 0) umma::tmem_dealloc(tmem, BWD_COLS);
}

}  // namespace w1tc

int launch_w1_finish(Workspace& w, int nparts, float* G, cudaStream_t s);   // nrm_w1.cu: sums the per-CTA partials in CTA order

template <int SPLIT>
static int launch_bwd(const float* P, Workspace& w, float* G, cudaStream_t s) {
  constexpr int NP = SPLIT == 3 ? 2 : 1;
  const size_t smem = sizeof(w1tc::SmemBwd<NP>);
  const long long ntiles = (w.NH + w1tc::ROWS - 1) / w1tc::ROWS;
  const int grid = (int)min(ntiles, (long long)min(sm_count(), W1_SPLITS));      // one CTA per SM (157 KB of shared memory), tiles in a grid-stride loop
  NRM_CUDA(cudaFuncSetAttribute(w1tc::w1_backward_tc_kernel<SPLIT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  launch_pdl(w1tc::w1_backward_tc_kernel<SPLIT>, dim3(grid), dim3(w1tc::BWD_THREADS), smem, s, w.xin_h, w.dxh, P, w.dxin_h, w.NH, w.splitk);
  NRM_LAUNCH_CHECK("w1_backward_tc_kernel");
  return launch_w1_finish(w, grid, G, s);
}
int launch_w1_backward_tc(const float* P, Workspace& w, float* G, int precision, cudaStream_t s) {
  return precision == NRM_PRECISION_BF16 ? launch_bwd<1>(P, w, G, s) : launch_bwd<3>(P, w, G, s);
}

}  // namespace nrm
