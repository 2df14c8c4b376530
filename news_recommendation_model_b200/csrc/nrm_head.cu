// BatchNorm1d(264) statistics of the scoring head (models/user_model.py:18,32): column sums of e_concat over the
// candidate rows, running-statistics update, and the BatchNorm part of the backward.  The six layers of the head
// themselves live in nrm_head_fused.cu.
#include "nrm_kernels.cuh"

namespace nrm {

// ---------------------------------------------------------------------------------
// BatchNorm statistics.  Column sums and sums of squares in double so that
// var = E[x^2] - mean^2 is safe (|mean| reaches 25 with var < 1 on some channels).
// ---------------------------------------------------------------------------------
__global__ void __launch_bounds__(E)
bn_partial_kernel(const float* __restrict__ e, long long R, int rows_per_chunk, double* __restrict__ part) {
  pdl_wait();                                          // programmatic dependent launch: see nrm_common.cuh
  pdl_trigger();
  const int n = threadIdx.x;
  const long long r0 = (long long)blockIdx.x * rows_per_chunk;
  const long long r1 = min(R, r0 + rows_per_chunk);
  double s = 0.0, q = 0.0;
#pragma unroll 8
  for (long long r = r0; r < r1; ++r) { const double v = (double)__ldg(e + r * E + n); s += v; q += v * v; }
  part[((long long)blockIdx.x * 2 + 0) * E + n] = s;
  part[((long long)blockIdx.x * 2 + 1) * E + n] = q;
}

// sums[i] = sum over parts of part[p][i], i < 2*264: one warp per sum, lane l adds parts l, l + 32, ... (all loads in
// flight at once), then a fixed shuffle tree.
__global__ void __launch_bounds__(256)
bn_partial_reduce_kernel(const double* __restrict__ part, int nparts, double* __restrict__ sums) {
  pdl_wait();                                          // programmatic dependent launch: see nrm_common.cuh
  pdl_trigger();
  const int i = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (i >= 2 * E) return;
  double s = 0.0;
#pragma unroll 8
  for (int p = lane; p < nparts; p += 32) s += part[(long long)p * 2 * E + i];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane == 0) sums[i] = s;
}

// de += rstd * gamma * (dz - mean_r(dz) - xhat * mean_r(dz * xhat))      (training)
// de += rstd * gamma * dz                                                 (eval)
// gate != null: `de` holds dx = dL/d(gate * e) as the tensor-core head backward leaves it; the direct path dx * gate is formed here
__global__ void __launch_bounds__(256)
bn_bwd_combine_kernel(const float* __restrict__ dz, const float* __restrict__ e, const float* __restrict__ mean,
                      const float* __restrict__ rstd, const float* __restrict__ gamma, const double* __restrict__ sums,
                      long long rows, int training, long long total4, const float* __restrict__ gate, float* __restrict__ de) {
  pdl_wait();                                          // programmatic dependent launch: see nrm_common.cuh
  pdl_trigger();
  // per-column means of dz and dz * xhat once per block (two double divisions per column instead of eight per element)
  __shared__ __align__(16) float s_m1[E], s_m2[E];
  if (training) {
    for (int n = threadIdx.x; n < E; n += 256) {
      s_m1[n] = (float)(sums[n] / (double)rows);
      s_m2[n] = (float)(sums[E + n] / (double)rows);
    }
    __syncthreads();
  }
  // four consecutive columns per thread (264 = 66 x 4: a float4 never straddles a row)
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < total4; i += (long long)gridDim.x * 256) {
    const int n = (int)(i % (E / 4)) * 4;
    const float4 rs = *reinterpret_cast<const float4*>(rstd + n), g = __ldg(reinterpret_cast<const float4*>(gamma + n));
    float4 v = __ldg(reinterpret_cast<const float4*>(dz) + i);
    if (training) {
      const float4 x = __ldg(reinterpret_cast<const float4*>(e) + i), mu = *reinterpret_cast<const float4*>(mean + n);
      const float4 m1 = *reinterpret_cast<const float4*>(s_m1 + n), m2 = *reinterpret_cast<const float4*>(s_m2 + n);
      v.x = v.x - m1.x - (x.x - mu.x) * rs.x * m2.x;
      v.y = v.y - m1.y - (x.y - mu.y) * rs.y * m2.y;
      v.z = v.z - m1.z - (x.z - mu.z) * rs.z * m2.z;
      v.w = v.w - m1.w - (x.w - mu.w) * rs.w * m2.w;
    }
    float4 d = reinterpret_cast<float4*>(de)[i];
    if (gate != nullptr) {
      const float4 gt = __ldg(reinterpret_cast<const float4*>(gate) + i);
      d.x *= gt.x; d.y *= gt.y; d.z *= gt.z; d.w *= gt.w;
    }
    d.x += rs.x * g.x * v.x; d.y += rs.y * g.y * v.y; d.z += rs.z * g.z * v.z; d.w += rs.w * g.w * v.w;
    reinterpret_cast<float4*>(de)[i] = d;
  }
}

// ---------------------------------------------------------------------------------
// launchers
// ---------------------------------------------------------------------------------
static inline int stat_rows(long long R) { return (int)((R + STAT_BLOCKS - 1) / STAT_BLOCKS); }
static inline int stat_chunks(long long R) { const int rp = stat_rows(R); return (int)((R + rp - 1) / rp); }

int launch_bn_partial_sums(Workspace& w, cudaStream_t s) {
  const int rp = stat_rows(w.R), nch = stat_chunks(w.R);
  launch_pdl(bn_partial_kernel, dim3(nch), dim3(E), 0, s, w.e, w.R, rp, w.stat_part);
  NRM_LAUNCH_CHECK("bn_partial_kernel");
  launch_pdl(bn_partial_reduce_kernel, dim3((2 * E + 7) / 8), dim3(256), 0, s, w.stat_part, nch, w.bn_sums);
  NRM_LAUNCH_CHECK("bn_partial_reduce_kernel");
  return NRM_OK;
}

int launch_bn_backward_combine(const float* P, Workspace& w, int training, const double* bn_bwd_sums,
                               long long global_rows, bool de_holds_dx, cudaStream_t s) {
  const long long total4 = w.R * (E / 4);
  const long long blocks = min((total4 + 255) / 256, (long long)sm_count() * 8);
  launch_pdl(bn_bwd_combine_kernel, dim3((int)blocks), dim3(256), 0, s, w.dz, w.e, w.mean, w.rstd, P + P_BN_W, bn_bwd_sums, global_rows, training, total4, de_holds_dx ? w.gate : nullptr, w.de);
  NRM_LAUNCH_CHECK("bn_bwd_combine_kernel");
  return NRM_OK;
}

}  // namespace nrm
