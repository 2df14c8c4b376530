// Shared definitions for libnrm_b200: flat parameter layout, workspace carving, small
// device helpers.  sm_100a only.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stddef.h>
#include <math.h>

#include "../../include/nrm_b200.h"

namespace nrm {

// ----------------------------------------------------------------------------
// problem constants (configs/model_config.py of the reference; SURVEY.md 3.3)
// ----------------------------------------------------------------------------
constexpr int D = 64;            // label-feature width == PCA width
constexpr int HC = 80;           // doubles per history row
constexpr int TC = 78;           // doubles per target row
constexpr int GC = 3;            // doubles per x_global row
constexpr int XIN = 66;          // w1 input width (56 feat + 8 time + read_time + scroll)
constexpr int E = 264;           // e_concat width  [eu_H 128 | eu_L 8 | ec 128]
constexpr int HID = 66;          // hidden width of the three head MLPs
constexpr int NCAT = 3000, NTYPE = 16, NYEAR = 100, NMONTH = 13, NDAY = 32, NHOUR = 24;
constexpr int NKEY32 = NCAT;                                   // keys of the 32-wide table
constexpr int K8_TYPE = 0, K8_YEAR = 16, K8_MONTH = 116, K8_DAY = 129, K8_HOUR = 161;
constexpr int NKEY8 = 185;                                     // keys of the 8-wide tables
constexpr float BN_EPS = 1e-5f;
constexpr float BN_MOMENTUM = 0.1f;

// e_concat column offsets
constexpr int E_LAB = 0, E_TI = 64, E_INST = 128, E_XT = 136, E_PCAT = 200;

// ----------------------------------------------------------------------------
// flat parameter layout (floats).  Order == reference state_dict order, delta last.
// Every entry starts on a 4-float (16 B) boundary; padding floats are kept at zero.
// ----------------------------------------------------------------------------
constexpr long long al4(long long x) { return (x + 3) & ~3LL; }
constexpr long long P_CAT = 0;
constexpr long long P_SENT_W = al4(P_CAT + NCAT * 32);
constexpr long long P_SENT_B = al4(P_SENT_W + 16 * 3);
constexpr long long P_TYPE = al4(P_SENT_B + 16);
constexpr long long P_W1_W = al4(P_TYPE + NTYPE * 8);
constexpr long long P_W1_B = al4(P_W1_W + 64 * XIN);
constexpr long long P_YEAR = al4(P_W1_B + 64);
constexpr long long P_MONTH = al4(P_YEAR + NYEAR * 8);
constexpr long long P_DAY = al4(P_MONTH + NMONTH * 8);
constexpr long long P_HOUR = al4(P_DAY + NDAY * 8);
constexpr long long P_LA_FC1_W = al4(P_HOUR + NHOUR * 8);
constexpr long long P_LA_FC1_B = al4(P_LA_FC1_W + 64 * 256);
constexpr long long P_LA_FC2_W = al4(P_LA_FC1_B + 64);
constexpr long long P_LA_FC2_B = al4(P_LA_FC2_W + 64);
constexpr long long P_TI_FC1_W = al4(P_LA_FC2_B + 1);
constexpr long long P_TI_FC1_B = al4(P_TI_FC1_W + 64 * 256);
constexpr long long P_TI_FC2_W = al4(P_TI_FC1_B + 64);
constexpr long long P_TI_FC2_B = al4(P_TI_FC2_W + 64);
constexpr long long P_INST_W = al4(P_TI_FC2_B + 1);
constexpr long long P_INST_B = al4(P_INST_W + 8 * 3);
constexpr long long P_BN_W = al4(P_INST_B + 8);
constexpr long long P_BN_B = al4(P_BN_W + E);
constexpr long long P_GATE_FC1_W = al4(P_BN_B + E);
constexpr long long P_GATE_FC1_B = al4(P_GATE_FC1_W + HID * E);
constexpr long long P_GATE_FC2_W = al4(P_GATE_FC1_B + HID);
constexpr long long P_GATE_FC2_B = al4(P_GATE_FC2_W + E * HID);
constexpr long long P_MLP_FC1_W = al4(P_GATE_FC2_B + E);
constexpr long long P_MLP_FC1_B = al4(P_MLP_FC1_W + HID * E);
constexpr long long P_MLP_FC2_W = al4(P_MLP_FC1_B + HID);
constexpr long long P_MLP_FC2_B = al4(P_MLP_FC2_W + E * HID);
constexpr long long P_OUT_FC1_W = al4(P_MLP_FC2_B + E);
constexpr long long P_OUT_FC1_B = al4(P_OUT_FC1_W + HID * E);
constexpr long long P_OUT_FC2_W = al4(P_OUT_FC1_B + HID);
constexpr long long P_OUT_FC2_B = al4(P_OUT_FC2_W + HID);
constexpr long long P_DELTA = al4(P_OUT_FC2_B + 1);      // == nrm_layout_fixed_floats()

// offsets of the four per-branch attention tensors relative to the branch base
struct AttOffsets { long long fc1_w, fc1_b, fc2_w, fc2_b; };
constexpr AttOffsets ATT_LABEL = {P_LA_FC1_W, P_LA_FC1_B, P_LA_FC2_W, P_LA_FC2_B};
constexpr AttOffsets ATT_TI = {P_TI_FC1_W, P_TI_FC1_B, P_TI_FC2_W, P_TI_FC2_B};

// ----------------------------------------------------------------------------
// error plumbing
// ----------------------------------------------------------------------------
void set_error(const char* fmt, ...);
int cuda_fail(cudaError_t e, const char* what);
#define NRM_CUDA(call)                                              \
  do {                                                              \
    cudaError_t e__ = (call);                                       \
    if (e__ != cudaSuccess) return ::nrm::cuda_fail(e__, #call);    \
  } while (0)
#define NRM_LAUNCH_CHECK(name)                                      \
  do {                                                              \
    ::nrm::count_launch();                                          \
    cudaError_t e__ = cudaGetLastError();                           \
    if (e__ != cudaSuccess) return ::nrm::cuda_fail(e__, name);     \
  } while (0)
// ----------------------------------------------------------------------------
// Programmatic dependent launch (PDL).  A kernel launched with launch_pdl() may begin (block scheduling, its code up to
// pdl_wait()) while the kernel in front of it on the stream is still draining, provided that kernel has executed
// pdl_trigger() in every block; pdl_wait() then blocks until the kernel in front has completed and its writes are
// visible.  Rules used here: every kernel launched with launch_pdl() executes pdl_wait() as its FIRST statement (so it
// never touches memory early) and pdl_trigger() right after it (the next kernel only ever waits at its own first
// statement).  Kernels in front that never trigger (torch's, memsets, NCCL) simply give the ordinary stream order.
// Works under stream capture (the edge becomes a programmatic graph dependency).  NRM_NO_PDL=1 disables the attribute.
// ----------------------------------------------------------------------------
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;\n" ::: "memory"); }
#ifdef NRM_PDL_EARLY_TRIGGER
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;\n" ::: "memory"); }
#else
__device__ __forceinline__ void pdl_trigger() {}      // implicit trigger when the block exits
#endif
bool pdl_enabled();
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl_enabled() ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

#define NRM_TRY(expr)            \
  do {                           \
    int rc__ = (expr);           \
    if (rc__ != NRM_OK) return rc__; \
  } while (0)

int sm_count();                      // of the current device
int current_device();
void count_launch();

// "Once per device" guard for cudaFuncSetAttribute-style set-up (function attributes are per device; a process may
// drive several GPUs from several threads).  first_time() is true for the callers that find the current device's flag clear;
// the flag is set right away, so two racing threads may both run the (idempotent) set-up, never neither.
struct DeviceOnce {
  unsigned char done[64] = {};
  bool first_time() {
    const int d = current_device();
    if (__atomic_load_n(&done[d], __ATOMIC_ACQUIRE)) return false;
    __atomic_store_n(&done[d], (unsigned char)1, __ATOMIC_RELEASE);
    return true;
  }
};

// Optional per-kernel device timing (nrm_timing_enable): brackets the launches issued
// during its lifetime with CUDA events on `stream`.  A no-op unless enabled.
struct KernelTimer {
  KernelTimer(const char* name, cudaStream_t stream);
  ~KernelTimer();
  int slot_; cudaStream_t stream_;
};

// ----------------------------------------------------------------------------
// workspace
// ----------------------------------------------------------------------------
constexpr int SORT_CHUNK = 2048;       // entries per counting-sort CTA
constexpr int SEG_GROUP = 128;         // sorted entries per level-1 segment group
constexpr int ATT_BWD_CTAS_MAX = 148;  // persistent grid of the attention backward
constexpr int ATT_PARTIAL = 3 * D * D + 64 + 64 + 4;   // dA | dWd | dBm | dw2 | db1 | db2 (+pad) floats per CTA
constexpr int ATT_TC_PARTS_MAX = 512; // CTAs of the tensor-core attention backward (2 per SM)
constexpr int ATT_TC_PARTIAL = 2 * 4096 + 68;   // dA^T | dWd^T | dw2 | db2 floats per CTA
constexpr int HEAD_WG_CHUNKS_MAX = 64; // row chunks of the head weight-gradient kernel
constexpr int STAT_BLOCKS = 256;       // row chunks of the column-statistics kernels
constexpr int HEAD_WT_W1T = 5 * HID * E;      // offset of w1.weight^T [66][64] in Workspace::head_wt (after the five head matrices)
constexpr int W1_SPLITS = 256;         // most CTAs (= partials) of the w1 backward

struct Workspace {
  // sizes
  int B, H, C;
  long long NH, R, N;                  // history rows, candidate rows, NH + R
  // forward (always)
  float* xin_h;        // [NH,66]   embedded history rows (w1 input)
  float* xh;           // [NH,64]   w1 output
  float* pca_h;        // [NH,64]   text/img PCA slice of the history rows as fp32
  float* e;            // [R,264]   e_concat
  float* mean;         // [264]
  float* rstd;         // [264]
  double* bn_sums;     // [2,264]   column sum / sum of squares of e
  double* stat_part;   // [STAT_BLOCKS,2,264]
  float* a1;           // [R,66]    gate.fc1 pre-activation
  float* gate;         // [R,264]
  float* a2;           // [R,66]    mlp.fc1 pre-activation
  float* y;            // [R,264]
  float* a3;           // [R,66]    out_mlp.fc1 pre-activation
  float* head_wt;      // [5][66*264] transposed head matrices (forward)
  float* head_part_f;  // [tiles][68]   out_mlp.fc2 partial gradients per row tile
  double* head_part_bn;// [tiles][2,264] BatchNorm backward partial sums per row tile
  float* head_part_w;  // [5][chunks][66*264+264] weight-gradient partials
  float* att_derived;  // [2][12420] derived attention weights (tensor-core paths)
  float* tp;           // [2][R,64]  tp = (Wb + Wc) t + b1 per candidate row and branch (tensor-core paths)
  unsigned char* att_dhid;  // label branch, training: dhid tile images (hi | lo) exported by the row-stacked backward for the input-gradient kernel
  float* att_sc;       // label branch, training: partial scores [tiles][4][128]
  unsigned int* head_arrive;   // arrival counter: the last CTA of the tensor-core head backward sums the BatchNorm partials
  float* head_img;     // operand images of the ten head products (nrm_head_tc.cu): bf16 parts, chunked in ring order
  float* att_rs_img;   // weight image of the row-stacked attention kernels (nrm_attention_rs.cu): bf16 operand tiles, hi | lo
  float* scores;       // caller's [2][B][C][H] attention scores (nrm_forward_scores; not carved: null = the forward stores none)
  // backward (training only)
  float* da3; float* da2; float* da1;   // [R,66]
  float* dy;           // [R,264]
  float* dgate;        // [R,264]
  float* de;           // [R,264]   dL/de (direct path, then + BN path)
  float* dz;           // [R,264]
  double* bn_bwd_sums; // [2,264]
  float* dxh;          // [NH,64]
  float* dxt;          // [R,64]
  float* dxin_h;       // [NH,66]
  float* att_part;     // [2][max(ATT_BWD_CTAS_MAX*ATT_PARTIAL, ATT_TC_PARTS_MAX*ATT_TC_PARTIAL)]
  float* dtp;          // [2][R,64]  dL/dtp per candidate row (tensor-core backward)
  float* att_dA;       // [2][64,64] summed dA per branch
  float* tp_part;      // [ceil(R/32)][4096+64] partial dBm | db1
  int att_tc_parts[2]; // CTAs (= partials) of the last tensor-core attention backward per branch (host side)
  float* splitk;       // [W1_SPLITS][64*66+64] per-CTA partials of the w1 gradients
  float* small_part;   // partial sums of the small reductions
  // sorted-segment machinery for the embedding-table gradients
  int* keys32;  int* keys8;            // [6N], [5N]
  int* perm32;  int* perm8;            // sorted entry -> entry id
  int* chunk_hist32; int* chunk_hist8; // [chunks][keys]
  int* seg32; int* seg8;               // per key: start[keys+1] | group_start[keys+1]
  int* gkey32; int* gkey8;             // group -> key
  float* gpart32; float* gpart8;       // [groups][W]
  size_t bytes;
};

// Carves `base` (may be null to only measure).  Returns total bytes.
size_t carve_workspace(Workspace& w, void* base, int B, int H, int C, int mode);

// ----------------------------------------------------------------------------
// device helpers
// ----------------------------------------------------------------------------
// Exact-erf GELU (nn.GELU() default of the reference, attention_model.py:21) and its derivative.
// Phi(x) = 0.5 (1 + erf(x / sqrt 2)) is evaluated with Abramowitz-Stegun 7.1.26:
//   erfc(z) = (a1 t + ... + a5 t^5) exp(-z^2),  t = 1 / (1 + p z),  z = |x| / sqrt 2,   |error| <= 1.5e-7,
// i.e. one MUFU.RCP + one MUFU.EX2 + 8 FMA-pipe operations instead of erff's ~35 instructions.
// Measured against float64 over [-12, 12] (tests/test_host_surface.py restates it in numpy):
// max |gelu error| 4.2e-7, max |gelu' error| 3.2e-7 -- below torch's own fp32 GELU error (1.2e-6).
// exp(-z^2) = exp(-x^2 / 2) is also sqrt(2 pi) times the normal pdf, so the derivative is free.
__device__ __forceinline__ float gelu_tail(float x, float& ex) {   // returns 0.5 * erfc(|x| / sqrt 2); ex = exp(-x^2 / 2)
  const float z = fabsf(x) * 0.70710678118654752440f;
  float t;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t) : "f"(fmaf(0.3275911f, z, 1.0f)));
  float poly = fmaf(t, 1.061405429f, -1.453152027f);
  poly = fmaf(t, poly, 1.421413741f);
  poly = fmaf(t, poly, -0.284496736f);
  poly = fmaf(t, poly, 0.254829592f);
  poly *= t;
  // exp(-x^2/2) = 2^(-w^2), w = |x| sqrt(log2(e) / 2): one multiply + ex2.approx.ftz (results below 2^-126, i.e. |x| > 13.2,
  // flush to zero) instead of __expf's range checks
  const float w = fabsf(x) * 0.84932180028801904272f;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(ex) : "f"(w * -w));
  return 0.5f * poly * ex;
}
__device__ __forceinline__ float gelu_f(float x) {
  float ex;
  const float half = gelu_tail(x, ex);
  return fmaf(-fabsf(x), half, fmaxf(x, 0.f));      // x >= 0: x (1 - half);  x < 0: x half
}
// returns gelu(x), writes d gelu / dx
__device__ __forceinline__ float gelu_both(float x, float& grad) {
  float ex;
  const float half = gelu_tail(x, ex);
  const float cdf = 0.5f + copysignf(0.5f - half, x);
  grad = fmaf(x * 0.39894228040143267794f, ex, cdf);
  return x * cdf;
}
__device__ __forceinline__ float gelu_grad_f(float x) {
  float g; (void)gelu_both(x, g); return g;
}
// ---- packed fp32 pairs (Blackwell fma.rn.f32x2 / mul / add): one issue slot for two FP32 operations.  The attention kernels are
// bound by issue slots on the CUDA cores (GELU, operand splits), so their element-wise math runs on pairs.
typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 pk(float a, float b) { f32x2 r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a), "f"(b)); return r; }
__device__ __forceinline__ void upk(f32x2 v, float& a, float& b) { asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v)); }
__device__ __forceinline__ f32x2 fma2(f32x2 a, f32x2 b, f32x2 c) { f32x2 d; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c)); return d; }
__device__ __forceinline__ f32x2 mul2(f32x2 a, f32x2 b) { f32x2 d; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
__device__ __forceinline__ f32x2 add2(f32x2 a, f32x2 b) { f32x2 d; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
// gelu(x) and d gelu / dx of a pair (same formulas as gelu_both):  q = 1/2 - 0.5 erfc(|x| / sqrt 2);  cdf = 1/2 + copysign(q, x);
// gelu = x cdf;  gelu' = cdf + x pdf,  pdf = exp(-x^2 / 2) / sqrt(2 pi)
__device__ __forceinline__ void gelu_both2(f32x2 x, f32x2& g, f32x2& gp) {
  float a, b, ta, tb, ea, eb;
  upk(x, a, b);
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(ta) : "f"(fmaf(fabsf(a), 0.23164189f, 1.0f)));
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(tb) : "f"(fmaf(fabsf(b), 0.23164189f, 1.0f)));
  upk(mul2(mul2(x, x), pk(-0.72134752044448170368f, -0.72134752044448170368f)), ea, eb);
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(ea) : "f"(ea));
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(eb) : "f"(eb));
  const f32x2 t2 = pk(ta, tb), e2 = pk(ea, eb);
  f32x2 poly = fma2(t2, pk(0.5f * 1.061405429f, 0.5f * 1.061405429f), pk(0.5f * -1.453152027f, 0.5f * -1.453152027f));
  poly = fma2(t2, poly, pk(0.5f * 1.421413741f, 0.5f * 1.421413741f));
  poly = fma2(t2, poly, pk(0.5f * -0.284496736f, 0.5f * -0.284496736f));
  poly = fma2(t2, poly, pk(0.5f * 0.254829592f, 0.5f * 0.254829592f));
  poly = mul2(poly, t2);
  float qa, qb;
  upk(fma2(poly, mul2(e2, pk(-1.f, -1.f)), pk(0.5f, 0.5f)), qa, qb);            // 1/2 - half >= 0
  const f32x2 cdf = add2(pk(copysignf(qa, a), copysignf(qb, b)), pk(0.5f, 0.5f));
  g = mul2(x, cdf);
  gp = fma2(mul2(x, pk(0.39894228040143267794f, 0.39894228040143267794f)), e2, cdf);
}

__device__ __forceinline__ int clampi(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }

}  // namespace nrm
