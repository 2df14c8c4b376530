// C ABI of libnrm_b200 (include/nrm_b200.h): argument checking, workspace carving and
// the kernel sequence of UserModel.forward / its backward.
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <vector>

#include "nrm_kernels.cuh"

namespace nrm {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
int cuda_fail(cudaError_t e, const char* what) {
  set_error("CUDA error %d (%s) at %s", (int)e, cudaGetErrorString(e), what);
  return NRM_ECUDA;
}
int current_device() {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 0;
  return dev;
}
int sm_count() {                      // per device (a process may drive several GPUs)
  static int n[64] = {};
  const int dev = current_device();
  int v = __atomic_load_n(&n[dev], __ATOMIC_RELAXED);
  if (v == 0) {
    if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || v <= 0) v = 148;
    __atomic_store_n(&n[dev], v, __ATOMIC_RELAXED);
  }
  return v;
}

// ---- launch counter and optional per-kernel event timing ------------------------------
static unsigned long long g_launches = 0;
void count_launch() { __atomic_fetch_add(&g_launches, 1ULL, __ATOMIC_RELAXED); }

constexpr int kTimerSlots = 40, kTimerRing = 256;
struct TimerSlot { const char* name; cudaEvent_t beg[kTimerRing], end[kTimerRing]; int used; bool made; };
static TimerSlot g_timers[kTimerSlots];
static int g_ntimers = 0;
static bool g_timing = false;
static std::mutex g_timer_mu;          // g_timers / g_ntimers (launches may come from several host threads)

KernelTimer::KernelTimer(const char* name, cudaStream_t stream) : slot_(-1), stream_(stream) {
  if (!g_timing) return;
  std::lock_guard<std::mutex> lock(g_timer_mu);
  int s = -1;
  for (int i = 0; i < g_ntimers; ++i) if (strcmp(g_timers[i].name, name) == 0) { s = i; break; }
  if (s < 0) { if (g_ntimers == kTimerSlots) return; s = g_ntimers++; g_timers[s].name = name; g_timers[s].used = 0; g_timers[s].made = false; }
  TimerSlot& t = g_timers[s];
  if (!t.made) { for (int i = 0; i < kTimerRing; ++i) { cudaEventCreate(&t.beg[i]); cudaEventCreate(&t.end[i]); } t.made = true; }
  if (t.used >= kTimerRing) return;
  slot_ = s;
  cudaEventRecord(t.beg[t.used], stream_);
}
KernelTimer::~KernelTimer() {
  if (slot_ < 0) return;
  std::lock_guard<std::mutex> lock(g_timer_mu);
  TimerSlot& t = g_timers[slot_];
  cudaEventRecord(t.end[t.used], stream_);
  t.used++;
}

// ---- side stream for work that only depends on the inputs ---------------------------------------
// The counting sort of the table ids needs nothing but the keys written by embed_rows_kernel, and its result is only
// used by the very last kernels of the backward.  It is enqueued on a library-owned side stream right after the
// embedding kernel (fork: event on the caller's stream) and joined just before the table-gradient kernels (join: event
// on the side stream), so its four small launches run under the attention / head kernels instead of after them.
// Fork and join are ordinary stream events, so the pattern is also valid inside a CUDA-graph capture of the caller's
// stream.
struct SideStream {
  int dev; cudaStream_t caller;
  cudaStream_t stream; cudaEvent_t fork, join, fork2, join2, fork0, join0, join_tp, fork3, join3, fork4, join4;
  // head weight gradients left for encoder_backward to enqueue on the side stream behind the w1 backward, i.e. beside the latency-bound
  // tail of the step (attention_finish, table gradients) instead of beside the attention backward kernels, which need whole SMs
  bool head_wgrad_pending = false; const float* wg_params = nullptr; float* wg_grads = nullptr; int wg_tiles = 0, wg_precision = 0;
};
// One side stream + event set per (device, caller stream): two models / threads that drive different streams of one device
// never share fork / join events (a wait can only ever bind to its own caller's record).  Created under a mutex on first use
// and kept for the life of the process (a caller that churns through streams leaks one small entry per stream).
static std::mutex g_side_mu;
static std::vector<SideStream*> g_sides;
static SideStream* side_stream(cudaStream_t caller) {
  const int dev = current_device();
  std::lock_guard<std::mutex> lock(g_side_mu);
  for (SideStream* p : g_sides)
    if (p->dev == dev && p->caller == caller) return p;
  SideStream* ss = new SideStream();
  ss->dev = dev; ss->caller = caller;
  bool ok = cudaStreamCreateWithFlags(&ss->stream, cudaStreamNonBlocking) == cudaSuccess;
  cudaEvent_t* evs[] = {&ss->fork, &ss->join, &ss->fork2, &ss->join2, &ss->fork0, &ss->join0, &ss->join_tp, &ss->fork3, &ss->join3,
                        &ss->fork4, &ss->join4};
  for (cudaEvent_t* e : evs) ok = ok && cudaEventCreateWithFlags(e, cudaEventDisableTiming) == cudaSuccess;
  if (!ok) { delete ss; return nullptr; }
  g_sides.push_back(ss);
  return ss;
}

bool pdl_enabled() {
  static const bool on = getenv("NRM_NO_PDL") == nullptr;
  return on;
}

struct LayoutEntry { const char* name; long long offset; long long numel; };
#define II "invariant_interest_model."
static const LayoutEntry kLayout[] = {
    {II "category_embedding.0.weight", P_CAT, NCAT * 32},
    {II "sentiment_embedding.0.weight", P_SENT_W, 16 * 3},
    {II "sentiment_embedding.0.bias", P_SENT_B, 16},
    {II "type_embedding.0.weight", P_TYPE, NTYPE * 8},
    {II "w1.weight", P_W1_W, 64 * XIN},
    {II "w1.bias", P_W1_B, 64},
    {II "year_embedding.0.weight", P_YEAR, NYEAR * 8},
    {II "month_embedding.0.weight", P_MONTH, NMONTH * 8},
    {II "day_embedding.0.weight", P_DAY, NDAY * 8},
    {II "hour_embedding.0.weight", P_HOUR, NHOUR * 8},
    {II "label_attention.mlp.fc1.weight", P_LA_FC1_W, 64 * 256},
    {II "label_attention.mlp.fc1.bias", P_LA_FC1_B, 64},
    {II "label_attention.mlp.fc2.weight", P_LA_FC2_W, 64},
    {II "label_attention.mlp.fc2.bias", P_LA_FC2_B, 1},
    {II "text_img_attention.mlp.fc1.weight", P_TI_FC1_W, 64 * 256},
    {II "text_img_attention.mlp.fc1.bias", P_TI_FC1_B, 64},
    {II "text_img_attention.mlp.fc2.weight", P_TI_FC2_W, 64},
    {II "text_img_attention.mlp.fc2.bias", P_TI_FC2_B, 1},
    {"instant_interest_model.out_fc.0.weight", P_INST_W, 8 * 3},
    {"instant_interest_model.out_fc.0.bias", P_INST_B, 8},
    {"bn.weight", P_BN_W, E},
    {"bn.bias", P_BN_B, E},
    {"gate.fc1.weight", P_GATE_FC1_W, HID * E},
    {"gate.fc1.bias", P_GATE_FC1_B, HID},
    {"gate.fc2.weight", P_GATE_FC2_W, E * HID},
    {"gate.fc2.bias", P_GATE_FC2_B, E},
    {"mlp.fc1.weight", P_MLP_FC1_W, HID * E},
    {"mlp.fc1.bias", P_MLP_FC1_B, HID},
    {"mlp.fc2.weight", P_MLP_FC2_W, E * HID},
    {"mlp.fc2.bias", P_MLP_FC2_B, E},
    {"out_mlp.fc1.weight", P_OUT_FC1_W, HID * E},
    {"out_mlp.fc1.bias", P_OUT_FC1_B, HID},
    {"out_mlp.fc2.weight", P_OUT_FC2_W, HID},
    {"out_mlp.fc2.bias", P_OUT_FC2_B, 1},
    {"delta", P_DELTA, -1},
};
#undef II
constexpr int kLayoutEntries = sizeof(kLayout) / sizeof(kLayout[0]);

size_t carve_workspace(Workspace& w, void* base, int B, int H, int C, int mode) {
  const bool training = (mode & NRM_MODE_KEEP_FOR_BWD) != 0;   // backward buffers wanted
  memset(&w, 0, sizeof(w));
  w.B = B; w.H = H; w.C = C;
  w.NH = (long long)B * H; w.R = (long long)B * C; w.N = w.NH + w.R;
  size_t off = 0;
  auto take = [&](size_t bytes) -> void* {
    void* p = base ? (char*)base + off : nullptr;
    off += (bytes + 255) & ~(size_t)255;
    return p;
  };
  const size_t f = sizeof(float);
  const size_t NH = (size_t)w.NH, R = (size_t)w.R, N = (size_t)w.N;
  w.xin_h = (float*)take(f * NH * XIN);
  w.xh = (float*)take(f * NH * 64);
  w.pca_h = (float*)take(f * NH * 64);
  w.e = (float*)take(f * R * E);
  w.mean = (float*)take(f * E);
  w.rstd = (float*)take(f * E);
  w.bn_sums = (double*)take(sizeof(double) * 2 * E);
  w.stat_part = (double*)take(sizeof(double) * STAT_BLOCKS * 2 * E);
  w.a1 = (float*)take(f * R * HID);
  w.gate = (float*)take(f * R * E);
  w.a2 = (float*)take(f * R * HID);
  w.y = (float*)take(f * R * E);
  w.a3 = (float*)take(f * R * HID);
  w.head_wt = (float*)take(f * (HEAD_WT_W1T + 64 * XIN));
  w.tp = (float*)take(f * 2 * R * 64);
  w.att_rs_img = (float*)take(attention_rs_image_bytes());
  w.head_img = (float*)take(head_tc_image_bytes());
  w.head_arrive = (unsigned int*)take(256);          // arrival counter of the tensor-core head backward (zeroed by the image kernel)
  if (training) {
    w.da3 = (float*)take(f * R * HID); w.da2 = (float*)take(f * R * HID); w.da1 = (float*)take(f * R * HID);
    w.dy = (float*)take(f * R * E);
    w.dgate = (float*)take(f * R * E);
    w.de = (float*)take(f * R * E);
    w.dz = (float*)take(f * R * E);
    w.bn_bwd_sums = (double*)take(sizeof(double) * 2 * E);
    w.head_part_f = (float*)take(f * ((R + 31) / 32) * 68);
    w.head_part_bn = (double*)take(sizeof(double) * ((R + 31) / 32) * 2 * E);
    w.head_part_w = (float*)take(f * 5 * HEAD_WG_CHUNKS_MAX * (HID * E + E));
    w.dxh = (float*)take(f * NH * 64);
    w.dxt = (float*)take(f * R * 64);
    w.dxin_h = (float*)take(f * NH * XIN);
    {
      const size_t ffma = (size_t)ATT_BWD_CTAS_MAX * ATT_PARTIAL, tc = (size_t)ATT_TC_PARTS_MAX * ATT_TC_PARTIAL;
      w.att_part = (float*)take(f * 2 * (ffma > tc ? ffma : tc));
    }
    w.dtp = (float*)take(f * 2 * R * 64);
    {
      const size_t tiles = (size_t)attention_rs_tiles(B, H, C);
      w.att_dhid = (unsigned char*)take(tiles * 2 * 16384);       // dhid tile images of the label branch (hi | lo)
      w.att_sc = (float*)take(f * tiles * 512);
    }
    w.att_dA = (float*)take(f * 2 * 4096);
    w.tp_part = (float*)take(f * 2 * ((R + 31) / 32) * (4096 + 64));
    w.splitk = (float*)take(f * (size_t)(64 * XIN + 64) * W1_SPLITS);   // per-CTA partials of the w1 weight / bias gradient
    w.small_part = (float*)take(f * 1024 * 96);
    const size_t n32 = N * 6, n8 = N * 5;
    const size_t c32 = (n32 + SORT_CHUNK - 1) / SORT_CHUNK, c8 = (n8 + SORT_CHUNK - 1) / SORT_CHUNK;
    const size_t g32 = n32 / SEG_GROUP + NKEY32 + 1, g8 = n8 / SEG_GROUP + NKEY8 + 1;
    w.keys32 = (int*)take(sizeof(int) * n32); w.keys8 = (int*)take(sizeof(int) * n8);
    w.perm32 = (int*)take(sizeof(int) * n32); w.perm8 = (int*)take(sizeof(int) * n8);
    w.chunk_hist32 = (int*)take(sizeof(int) * c32 * NKEY32); w.chunk_hist8 = (int*)take(sizeof(int) * c8 * NKEY8);
    w.seg32 = (int*)take(sizeof(int) * 3 * (NKEY32 + 1)); w.seg8 = (int*)take(sizeof(int) * 3 * (NKEY8 + 1));   // starts | group starts | totals
    w.gkey32 = (int*)take(sizeof(int) * g32); w.gkey8 = (int*)take(sizeof(int) * g8);
    w.gpart32 = (float*)take(f * g32 * 32); w.gpart8 = (float*)take(f * g8 * 8);
  }
  w.bytes = off;
  return off;
}

static int check_shape(const char* fn, int B, int H, int C) {
  if (B <= 0 || H <= 0 || C <= 0) { set_error("%s: B, H, C must be positive (got %d, %d, %d)", fn, B, H, C); return NRM_EINVAL; }
  if (((long long)B * H + (long long)B * C) * 6 >= (1LL << 31)) { set_error("%s: batch too large for 32-bit entry ids", fn); return NRM_EINVAL; }
  return NRM_OK;
}
static int get_workspace(const char* fn, Workspace& w, void* ws, size_t ws_bytes, int B, int H, int C, int mode) {
  if (ws == nullptr || ((uintptr_t)ws & 255) != 0) { set_error("%s: workspace must be non-null and 256-byte aligned", fn); return NRM_EWORKSPACE; }
  const size_t need = carve_workspace(w, ws, B, H, C, mode);
  if (need > ws_bytes) { set_error("%s: workspace too small (%zu < %zu bytes)", fn, ws_bytes, need); return NRM_EWORKSPACE; }
  return NRM_OK;
}

static int encoder_forward(const BatchPtrs& in, const float* P, Workspace& w, int mode, int precision, cudaStream_t s) {
  SideStream* ss = side_stream(s);
  if (ss == nullptr) { set_error("encoder_forward: cannot create the side stream"); return NRM_ECUDA; }
  const bool tc = precision != NRM_PRECISION_FP32;
  // fork 0: what depends on the weights only (transposed head matrices, the operand images of the tensor-core attention and head)
  // runs on the side stream under the embedding kernel
  NRM_CUDA(cudaEventRecord(ss->fork0, s));
  NRM_CUDA(cudaStreamWaitEvent(ss->stream, ss->fork0, 0));
  NRM_TRY(launch_head_transpose(P, w, ss->stream));          // includes w1^T for the history projection below
  NRM_CUDA(cudaEventRecord(ss->join0, ss->stream));
  if (tc) {
    NRM_TRY(launch_attention_prep_rs(P, w, ss->stream));
    NRM_TRY(launch_head_images_tc(P, w, precision, (mode & NRM_MODE_KEEP_FOR_BWD) != 0, ss->stream));
  }
  { KernelTimer t("embed_rows", s);
    NRM_TRY(launch_embed_rows(in, P, w, (mode & NRM_MODE_KEEP_FOR_BWD) != 0, s)); }
  // fork: the per-candidate vectors tp (they need the candidate rows of e) run under the w1 projection; then, for the
  // backward's table gradients, the sort of the table ids (joined in encoder_backward)
  NRM_CUDA(cudaEventRecord(ss->fork, s));
  NRM_CUDA(cudaStreamWaitEvent(ss->stream, ss->fork, 0));
  if (tc) NRM_TRY(launch_candidate_tp(P, w, ss->stream));
  NRM_CUDA(cudaEventRecord(ss->join_tp, ss->stream));
  if (mode & NRM_MODE_KEEP_FOR_BWD) {
    NRM_TRY(launch_table_sort(w, ss->stream));
    NRM_CUDA(cudaEventRecord(ss->join, ss->stream));
  }
  // xh = w1(xin_h)   (user_invariant_interest_model.py:78)
  NRM_CUDA(cudaStreamWaitEvent(s, ss->join0, 0));            // w1^T ready
  { KernelTimer t("w1_forward", s); NRM_TRY(launch_w1_forward(P, w, s)); }
  NRM_CUDA(cudaStreamWaitEvent(s, ss->join_tp, 0));          // join: operand images, transposed head matrices, tp
  if (!tc) {
    { KernelTimer t("attention_forward_label", s); NRM_TRY(launch_attention_forward(P, w, 0, s)); }
    { KernelTimer t("attention_forward_textimg", s); NRM_TRY(launch_attention_forward(P, w, 1, s)); }
  } else {
    // tensor-core path: one launch covers both branches
    KernelTimer t("attention_forward", s);
    NRM_TRY(launch_attention_forward_rs(w, precision, s));
  }
  // join: the id sort (long finished: it ran under the w1 / attention kernels) comes back to the caller's stream HERE, so a
  // training-mode forward that is never followed by a backward (validation with gradients enabled, a graph capture of the
  // forward alone) leaves no unjoined side-stream work, and the workspace may be reused or freed in stream order
  if (mode & NRM_MODE_KEEP_FOR_BWD) NRM_CUDA(cudaStreamWaitEvent(s, ss->join, 0));
  return NRM_OK;
}

static int encoder_backward(const BatchPtrs& in, const float* P, Workspace& w, int precision, float* G, cudaStream_t s) {
  SideStream* ss = side_stream(s);
  if (ss == nullptr) { set_error("encoder_backward: cannot create the side stream"); return NRM_ECUDA; }
  const bool tc = precision != NRM_PRECISION_FP32;
  // tensor-core precisions: the row-stacked backward sums over rows (weight gradients, dtp); its label branch exports dhid for the
  // input-gradient kernel
  { KernelTimer t("attention_backward_label", s);
    if (tc) NRM_TRY(launch_attention_backward_rs(w, 0, precision, true, s)); else NRM_TRY(launch_attention_backward(P, w, 0, s)); }
  if (tc) {
    // the label branch's input gradients (dxh, dxt) come from the dhid tiles the kernel above exported
    KernelTimer t("attention_input_grad_label", s);
    NRM_TRY(launch_attention_input_grad_rs(w, precision, s));
  }
  // fork: the w1 backward only needs dxh (label attention).  The text/img attention backward is launched FIRST: both become ready
  // when the input-gradient kernel ends, both want every SM (one CTA of 150-200 KB each), and the one launched first gets them -- the
  // attention kernel is on the critical path, the w1 backward then runs beside attention_finish in the latency-bound tail
  NRM_CUDA(cudaEventRecord(ss->fork2, s));
  NRM_CUDA(cudaStreamWaitEvent(ss->stream, ss->fork2, 0));
  { KernelTimer t("attention_backward_textimg", s);
    if (tc) NRM_TRY(launch_attention_backward_rs(w, 1, precision, false, s)); else NRM_TRY(launch_attention_backward(P, w, 1, s)); }
  // w1: dxin_h = dxh W1, dW1 = dxh^T xin_h, db1 = colsum(dxh)
  { KernelTimer t("w1_backward", ss->stream);
    if (tc) NRM_TRY(launch_w1_backward_tc(P, w, G, precision, ss->stream)); else NRM_TRY(launch_w1_backward(P, w, G, ss->stream)); }
  NRM_CUDA(cudaEventRecord(ss->join2, ss->stream));
  if (ss->head_wgrad_pending) {                              // behind the w1 backward on the side stream; covered by join3 below
    ss->head_wgrad_pending = false;
    KernelTimer t("head_wgrad", ss->stream);
    NRM_TRY(launch_head_backward_wgrad(ss->wg_params, w, ss->wg_grads, ss->stream, ss->wg_tiles, ss->wg_precision));
  }
  { KernelTimer t("attention_finish", s);
    if (tc) NRM_TRY(launch_attention_finish_tc(P, w, G, s));   // one pass for both branches
    else { NRM_TRY(launch_attention_finish(P, w, 0, G, s)); NRM_TRY(launch_attention_finish(P, w, 1, G, s)); } }
  NRM_CUDA(cudaStreamWaitEvent(s, ss->join2, 0));          // join: dxin_h ready
  // fork: the sentiment / instant Linear gradients (side stream) next to the table gradients (two latency-bound kernel
  // pairs that write disjoint gradient ranges)
  NRM_CUDA(cudaEventRecord(ss->fork3, s));
  NRM_CUDA(cudaStreamWaitEvent(ss->stream, ss->fork3, 0));
  { KernelTimer t("small_linear_grads", ss->stream); NRM_TRY(launch_small_linear_grads(in, w, G, ss->stream)); }
  NRM_CUDA(cudaEventRecord(ss->join3, ss->stream));
  // (the id sort enqueued by the forward was joined at the end of that forward)
  NRM_TRY(launch_table_grads(w, G, s));
  NRM_CUDA(cudaStreamWaitEvent(s, ss->join3, 0));
  return NRM_OK;
}

}  // namespace nrm

using namespace nrm;

extern "C" int nrm_version(void) { return 100; }
extern "C" unsigned long long nrm_launch_count(void) { return __atomic_load_n(&g_launches, __ATOMIC_RELAXED); }
extern "C" void nrm_timing_enable(int on) {
  std::lock_guard<std::mutex> lock(g_timer_mu);
  g_timing = on != 0;
  for (int i = 0; i < g_ntimers; ++i) g_timers[i].used = 0;
}
// Writes "name count total_ms\n" lines for every timed kernel group; synchronises the events.
extern "C" int nrm_timing_report(char* buf, size_t buf_bytes) {
  if (!buf || buf_bytes == 0) { set_error("nrm_timing_report: bad buffer"); return NRM_EINVAL; }
  size_t off = 0;
  buf[0] = 0;
  std::lock_guard<std::mutex> lock(g_timer_mu);
  for (int i = 0; i < g_ntimers; ++i) {
    TimerSlot& t = g_timers[i];
    double total = 0.0;
    for (int k = 0; k < t.used; ++k) {
      float ms = 0.f;
      NRM_CUDA(cudaEventSynchronize(t.end[k]));
      NRM_CUDA(cudaEventElapsedTime(&ms, t.beg[k], t.end[k]));
      total += ms;
    }
    // optional 4th / 5th columns: start and end of the group's LAST recorded launch relative to the first event of the first group
    // (a timeline: gaps and overlaps between groups, tools/step_timeline.py)
    float t_beg = 0.f, t_end = 0.f;
    if (t.used > 0 && g_ntimers > 0 && g_timers[0].used > 0) {
      cudaEventElapsedTime(&t_beg, g_timers[0].beg[g_timers[0].used - 1], t.beg[t.used - 1]);
      cudaEventElapsedTime(&t_end, g_timers[0].beg[g_timers[0].used - 1], t.end[t.used - 1]);
    }
    const int n = snprintf(buf + off, buf_bytes - off, "%s %d %.6f %.6f %.6f\n", t.name, t.used, total, t_beg, t_end);
    if (n < 0 || (size_t)n >= buf_bytes - off) break;
    off += (size_t)n;
  }
  return NRM_OK;
}
// per-role wait cycles of the row-stacked attention kernels (development builds with -DNRM_RS_PROFILE); reads and clears
extern "C" int nrm_debug_rsprof(long long* host_out64) { return rsprof_read(host_out64); }
// Byte offset / size of a named workspace buffer (debugging aid: lets a script compare intermediate buffers between runs)
extern "C" long long nrm_debug_ws_field(int B, int H, int C, int mode, const char* name, long long* bytes) {
  if (B <= 0 || H <= 0 || C <= 0 || !name || !bytes) return -1;
  Workspace w;
  carve_workspace(w, reinterpret_cast<void*>(uintptr_t(256)), B, H, C, mode);
  const size_t R = (size_t)w.R, NH = (size_t)w.NH;
  struct F { const char* n; const void* p; size_t b; };
  const F fields[] = {{"e", w.e, R * E * 4}, {"de", w.de, R * E * 4}, {"dz", w.dz, R * E * 4}, {"dxh", w.dxh, NH * 64 * 4}, {"dxt", w.dxt, R * 64 * 4},
                      {"dxin_h", w.dxin_h, NH * XIN * 4}, {"att_dhid", w.att_dhid, (size_t)attention_rs_tiles(B, H, C) * 2 * 16384},
                      {"att_sc", w.att_sc, (size_t)attention_rs_tiles(B, H, C) * 512 * 4}, {"xh", w.xh, NH * 64 * 4}, {"dtp", w.dtp, 2 * R * 64 * 4},
                      {"tp", w.tp, 2 * R * 64 * 4}};
  for (const F& f : fields)
    if (strcmp(f.n, name) == 0 && f.p != nullptr) { *bytes = (long long)f.b; return (long long)(reinterpret_cast<uintptr_t>(f.p) - 256); }
  return -1;
}
extern "C" int nrm_debug_headprof(long long* host_out32) { return headprof_read(host_out32); }
extern "C" const char* nrm_last_error(void) { return g_err; }
extern "C" int nrm_layout_entries(void) { return kLayoutEntries; }
extern "C" const char* nrm_layout_name(int i) { return (i >= 0 && i < kLayoutEntries) ? kLayout[i].name : nullptr; }
extern "C" long long nrm_layout_offset(int i) { return (i >= 0 && i < kLayoutEntries) ? kLayout[i].offset : -1; }
extern "C" long long nrm_layout_numel(int i) { return (i >= 0 && i < kLayoutEntries) ? kLayout[i].numel : -1; }
extern "C" long long nrm_layout_fixed_floats(void) { return P_DELTA; }

extern "C" size_t nrm_workspace_bytes(int B, int H, int C, int mode) {
  if (B <= 0 || H <= 0 || C <= 0) return 0;
  Workspace w;
  return carve_workspace(w, nullptr, B, H, C, mode);
}

// Byte offset of e_concat [R,264] inside a workspace carved for (B, H, C, mode): lets a caller of nrm_forward_encoder read the
// encoder output (eu_H | eu_L | ec) without knowing the carve order.
extern "C" size_t nrm_workspace_e_offset(int B, int H, int C, int mode) {
  if (B <= 0 || H <= 0 || C <= 0) return 0;
  Workspace w;
  carve_workspace(w, reinterpret_cast<void*>(uintptr_t(256)), B, H, C, mode);
  return (size_t)(reinterpret_cast<uintptr_t>(w.e) - 256);
}

// scores non-null: the attention kernels also export s_label / s_ti there (eval-mode forwards, nrm_forward_scores)
static int forward_encoder_impl(const char* fn, const BatchPtrs& in, int B, int H, int C, const float* params, int mode, int precision,
                                double* bn_sums, float* scores, void* workspace, size_t workspace_bytes, void* stream) {
  Workspace w;
  NRM_TRY(get_workspace(fn, w, workspace, workspace_bytes, B, H, C, mode));
  w.scores = scores;
  cudaStream_t s = (cudaStream_t)stream;
  NRM_TRY(encoder_forward(in, params, w, mode, precision, s));
  if (mode & NRM_MODE_BN_BATCH_STATS) {
    KernelTimer t("bn_statistics", s);
    NRM_TRY(launch_bn_partial_sums(w, s));
    if (bn_sums != nullptr && bn_sums != w.bn_sums)
      NRM_CUDA(cudaMemcpyAsync(bn_sums, w.bn_sums, sizeof(double) * 2 * E, cudaMemcpyDeviceToDevice, s));
  }
  return NRM_OK;
}

// packed float64 rows from the caller: one impression's rows are dense, the batch stride may be larger
static int packed_batch(const char* fn, const double* x_history, const double* x_target, long long xt_bs, const double* x_global,
                        long long xg_bs, int C, BatchPtrs& in) {
  if (!x_history || !x_target || !x_global) { set_error("%s: null pointer", fn); return NRM_EINVAL; }
  if (xt_bs < (long long)C * TC || xg_bs < (long long)C * GC) { set_error("%s: batch stride smaller than one impression", fn); return NRM_EINVAL; }
  in = BatchPtrs{x_history, x_target, xt_bs, x_global, xg_bs};
  return NRM_OK;
}

// compact wire format as the input of the row kernels (no expansion to the packed float64 tensors); cand_bs: the batch stride of the
// candidate ids, C, or 0 when every impression has the same candidates
static int compact_batch(const char* fn, const nrm_compact_batch* cb, int cand_bs, BatchPtrs& in) {
  if (!cb || !cb->articles || cb->n_articles <= 0 || !cb->hist_article || !cb->hist_time || !cb->hist_click || !cb->cand_article || !cb->cand_time) {
    set_error("%s: bad compact batch", fn); return NRM_EINVAL;
  }
  if ((reinterpret_cast<uintptr_t>(cb->articles) & 15) != 0) { set_error("%s: the article table must be 16-byte aligned", fn); return NRM_EINVAL; }
  if (cb->label32 && !cb->label64) { set_error("%s: bad compact batch", fn); return NRM_EINVAL; }
  in = BatchPtrs{};
  in.compact = CompactPtrs{cb->articles, cb->n_articles, cand_bs, cb->hist_article, cb->hist_time, cb->hist_click, cb->cand_article,
                           cb->cand_time, cb->label32, cb->label64};
  return NRM_OK;
}

extern "C" int nrm_forward_encoder(const double* x_history, const double* x_target, long long xt_bs, const double* x_global,
                                   long long xg_bs, int B, int H, int C, const float* params, int mode, int precision,
                                   double* bn_sums, void* workspace, size_t workspace_bytes, void* stream) {
  const char* fn = "nrm_forward_encoder";
  NRM_TRY(check_shape(fn, B, H, C));
  BatchPtrs in;
  NRM_TRY(packed_batch(fn, x_history, x_target, xt_bs, x_global, xg_bs, C, in));
  if (!params) { set_error("%s: null pointer", fn); return NRM_EINVAL; }
  return forward_encoder_impl(fn, in, B, H, C, params, mode, precision, bn_sums, nullptr, workspace, workspace_bytes, stream);
}

extern "C" int nrm_forward_encoder_compact(const nrm_compact_batch* batch, int B, int H, int C, const float* params, int mode, int precision,
                                           double* bn_sums, void* workspace, size_t workspace_bytes, void* stream) {
  const char* fn = "nrm_forward_encoder_compact";
  NRM_TRY(check_shape(fn, B, H, C));
  if (!params) { set_error("%s: null pointer", fn); return NRM_EINVAL; }
  BatchPtrs in;
  NRM_TRY(compact_batch(fn, batch, C, in));
  return forward_encoder_impl(fn, in, B, H, C, params, mode, precision, bn_sums, nullptr, workspace, workspace_bytes, stream);
}

extern "C" int nrm_forward_head(int B, int H, int C, const float* params, float* bn_running_mean, float* bn_running_var,
                                  long long* bn_num_batches_tracked, int mode, int precision, const double* bn_sums,
                                  long long bn_global_rows, float* logits, void* workspace, size_t workspace_bytes,
                                  void* stream) {
  const int training = mode & NRM_MODE_BN_BATCH_STATS;
  NRM_TRY(check_shape("nrm_forward_head", B, H, C));
  if (!params || !bn_running_mean || !bn_running_var || !logits) { set_error("nrm_forward_head: null pointer"); return NRM_EINVAL; }
  if (training && !bn_num_batches_tracked) { set_error("nrm_forward_head: null num_batches_tracked"); return NRM_EINVAL; }
  Workspace w;
  NRM_TRY(get_workspace("nrm_forward_head", w, workspace, workspace_bytes, B, H, C, mode));
  const double* sums = bn_sums ? bn_sums : w.bn_sums;
  const long long rows = bn_global_rows > 0 ? bn_global_rows : w.R;
  KernelTimer t("head_forward", (cudaStream_t)stream);
  if (precision != NRM_PRECISION_FP32)
    return launch_head_forward_tc(params, w, precision, bn_running_mean, bn_running_var, bn_num_batches_tracked, training,
                                  (mode & NRM_MODE_KEEP_FOR_BWD) != 0, sums, rows, logits, (cudaStream_t)stream);
  // the BatchNorm finalisation (batch / running statistics, running-statistics update) is the prologue of the fused kernel
  return launch_head_forward_fused(params, w, bn_running_mean, bn_running_var, bn_num_batches_tracked, training,
                                   (mode & NRM_MODE_KEEP_FOR_BWD) != 0, sums, rows, logits, (cudaStream_t)stream);
}

extern "C" int nrm_forward(const double* x_history, const double* x_target, long long xt_bs, const double* x_global,
                           long long xg_bs, int B, int H, int C, const float* params, float* bn_running_mean,
                           float* bn_running_var, long long* bn_num_batches_tracked, int mode, int precision,
                           float* logits, void* workspace, size_t workspace_bytes, void* stream) {
  NRM_TRY(nrm_forward_encoder(x_history, x_target, xt_bs, x_global, xg_bs, B, H, C, params, mode, precision, nullptr,
                              workspace, workspace_bytes, stream));
  return nrm_forward_head(B, H, C, params, bn_running_mean, bn_running_var, bn_num_batches_tracked, mode, precision, nullptr, 0,
                            logits, workspace, workspace_bytes, stream);
}

extern "C" int nrm_forward_compact(const nrm_compact_batch* batch, int B, int H, int C, const float* params, float* bn_running_mean,
                                   float* bn_running_var, long long* bn_num_batches_tracked, int mode, int precision,
                                   float* logits, void* workspace, size_t workspace_bytes, void* stream) {
  NRM_TRY(nrm_forward_encoder_compact(batch, B, H, C, params, mode, precision, nullptr, workspace, workspace_bytes, stream));
  return nrm_forward_head(B, H, C, params, bn_running_mean, bn_running_var, bn_num_batches_tracked, mode, precision, nullptr, 0,
                            logits, workspace, workspace_bytes, stream);
}

// ---- attention scores (explanations): eval-mode forward that also exports s_label / s_ti -----------------------------------------
static int scores_args(const char* fn, int mode, const float* scores) {
  if (mode != NRM_MODE_EVAL) { set_error("%s: scores are exported by eval-mode forwards only (mode must be NRM_MODE_EVAL, got %d)", fn, mode); return NRM_EINVAL; }
  if (!scores) { set_error("%s: null scores", fn); return NRM_EINVAL; }
  return NRM_OK;
}

extern "C" int nrm_forward_scores(const double* x_history, const double* x_target, long long xt_bs, const double* x_global,
                                  long long xg_bs, int B, int H, int C, const float* params, float* bn_running_mean,
                                  float* bn_running_var, long long* bn_num_batches_tracked, int mode, int precision,
                                  float* logits, float* scores, void* workspace, size_t workspace_bytes, void* stream) {
  const char* fn = "nrm_forward_scores";
  NRM_TRY(check_shape(fn, B, H, C));
  BatchPtrs in;
  NRM_TRY(packed_batch(fn, x_history, x_target, xt_bs, x_global, xg_bs, C, in));
  if (!params) { set_error("%s: null pointer", fn); return NRM_EINVAL; }
  NRM_TRY(scores_args(fn, mode, scores));
  NRM_TRY(forward_encoder_impl(fn, in, B, H, C, params, mode, precision, nullptr, scores, workspace, workspace_bytes, stream));
  return nrm_forward_head(B, H, C, params, bn_running_mean, bn_running_var, bn_num_batches_tracked, mode, precision, nullptr, 0,
                          logits, workspace, workspace_bytes, stream);
}

extern "C" int nrm_forward_scores_compact(const nrm_compact_batch* batch, int B, int H, int C, const float* params, float* bn_running_mean,
                                          float* bn_running_var, long long* bn_num_batches_tracked, int mode, int precision,
                                          float* logits, float* scores, void* workspace, size_t workspace_bytes, void* stream) {
  const char* fn = "nrm_forward_scores_compact";
  NRM_TRY(check_shape(fn, B, H, C));
  if (!params) { set_error("%s: null pointer", fn); return NRM_EINVAL; }
  BatchPtrs in;
  NRM_TRY(compact_batch(fn, batch, C, in));
  NRM_TRY(scores_args(fn, mode, scores));
  NRM_TRY(forward_encoder_impl(fn, in, B, H, C, params, mode, precision, nullptr, scores, workspace, workspace_bytes, stream));
  return nrm_forward_head(B, H, C, params, bn_running_mean, bn_running_var, bn_num_batches_tracked, mode, precision, nullptr, 0,
                          logits, workspace, workspace_bytes, stream);
}

// ---- recommendation from a shared pool: every user against the same N articles, in chunks of the pool ------------------------------
// Workspace: the chunk's [B,C] logits and the eval workspace of a (B, H, C) forward.  The row kernels read the users' compact histories
// as they are and the chunk's candidate ids with batch stride 0, so all B users see the same candidates without a copy per user.  C is
// a multiple of 8, the row-stacked attention's candidate group (rs::CG), so every chunk groups candidates exactly as one forward over
// all N columns would: the logits are that forward's, bit for bit.
struct PoolCarve { float* out; void* ws; size_t ws_bytes, bytes; };
static void carve_pool(PoolCarve& pc, void* base, int B, int H, int N, int chunk) {
  const int C = chunk < N ? chunk : N;
  size_t off = 0;
  auto take = [&](size_t bytes) -> void* {
    void* p = base ? (char*)base + off : nullptr;
    off += (bytes + 255) & ~(size_t)255;
    return p;
  };
  pc.out = (float*)take(sizeof(float) * B * C);
  Workspace w;
  pc.ws_bytes = carve_workspace(w, nullptr, B, H, C, NRM_MODE_EVAL);
  pc.ws = take(pc.ws_bytes);
  pc.bytes = off;
}

extern "C" size_t nrm_pool_workspace_bytes(int B, int H, int N, int chunk) {
  if (B <= 0 || H <= 0 || N <= 0 || chunk <= 0) return 0;
  PoolCarve pc;
  carve_pool(pc, nullptr, B, H, N, chunk);
  return pc.bytes;
}

extern "C" int nrm_forward_pool(const nrm_compact_batch* users, int B, int H, int N, int chunk, const float* params,
                                const float* bn_running_mean, const float* bn_running_var, int precision, float* logits,
                                void* workspace, size_t workspace_bytes, void* stream) {
  const char* fn = "nrm_forward_pool";
  if (B <= 0 || H <= 0 || N <= 0) { set_error("%s: B, H, N must be positive (got %d, %d, %d)", fn, B, H, N); return NRM_EINVAL; }
  if (chunk <= 0 || chunk % 8 != 0) { set_error("%s: chunk must be a positive multiple of 8 (got %d)", fn, chunk); return NRM_EINVAL; }
  if (precision < NRM_PRECISION_FP32 || precision > NRM_PRECISION_BF16X3) { set_error("%s: unknown precision %d", fn, precision); return NRM_EINVAL; }
  BatchPtrs in;
  NRM_TRY(compact_batch(fn, users, 0, in));
  if (users->label32 || users->label64) { set_error("%s: the pool has no labels (label32 / label64 must be null)", fn); return NRM_EINVAL; }
  if (!params || !bn_running_mean || !bn_running_var || !logits) { set_error("%s: null pointer", fn); return NRM_EINVAL; }
  const int C = chunk < N ? chunk : N;
  NRM_TRY(check_shape(fn, B, H, C));
  if (workspace == nullptr || ((uintptr_t)workspace & 255) != 0) { set_error("%s: workspace must be non-null and 256-byte aligned", fn); return NRM_EWORKSPACE; }
  PoolCarve pc;
  carve_pool(pc, workspace, B, H, N, chunk);
  if (pc.bytes > workspace_bytes) { set_error("%s: workspace too small (%zu < %zu bytes)", fn, workspace_bytes, pc.bytes); return NRM_EWORKSPACE; }
  cudaStream_t s = (cudaStream_t)stream;
  // the BatchNorm buffers are only read in eval mode: the head's training-only writes never happen
  float* run_mean = const_cast<float*>(bn_running_mean);
  float* run_var = const_cast<float*>(bn_running_var);
  for (int c0 = 0; c0 < N; c0 += C) {
    const int nc = N - c0 < C ? N - c0 : C;
    BatchPtrs chunk_in = in;
    chunk_in.compact.cand_article += c0; chunk_in.compact.cand_time += c0;
    NRM_TRY(forward_encoder_impl(fn, chunk_in, B, H, nc, params, NRM_MODE_EVAL, precision, nullptr, nullptr, pc.ws, pc.ws_bytes, stream));
    float* out = nc == N ? logits : pc.out;                 // a single chunk writes the [B,N] logits directly
    NRM_TRY(nrm_forward_head(B, H, nc, params, run_mean, run_var, nullptr, NRM_MODE_EVAL, precision, nullptr, 0, out, pc.ws, pc.ws_bytes, stream));
    if (out != logits)
      NRM_CUDA(cudaMemcpy2DAsync(logits + c0, sizeof(float) * N, out, sizeof(float) * nc, sizeof(float) * nc, B, cudaMemcpyDeviceToDevice, s));
  }
  return NRM_OK;
}

// head data gradients down to w.de and the BatchNorm backward sums: one tensor-core chain, or the FFMA dgrad + BatchNorm pass
static int head_dgrad(const float* params, Workspace& w, int precision, const float* dlogits, float* grads, cudaStream_t s) {
  if (precision != NRM_PRECISION_FP32) return launch_head_backward_dgrad_tc(params, w, precision, dlogits, grads, s);
  NRM_TRY(launch_head_backward_dgrad(params, w, dlogits, s));
  return launch_head_backward_bn(w, grads, s, 0);
}

// defer_wgrad: the head's weight gradients (only the optimizer needs them) are left to the next encoder backward on this stream, which
// enqueues them on the side stream behind the w1 backward, beside its own tail, instead of in front of it
static int backward_head(const char* fn, bool defer_wgrad, int B, int H, int C, const float* params, int precision, const float* dlogits, float* grads,
                         double* bn_bwd_sums, void* workspace, size_t workspace_bytes, void* stream) {
  NRM_TRY(check_shape(fn, B, H, C));
  if (!params || !dlogits || !grads) { set_error("%s: null pointer", fn); return NRM_EINVAL; }
  Workspace w;
  NRM_TRY(get_workspace(fn, w, workspace, workspace_bytes, B, H, C, NRM_MODE_KEEP_FOR_BWD));
  cudaStream_t s = (cudaStream_t)stream;
  const bool tc = precision != NRM_PRECISION_FP32;
  const int tiles = tc ? head_tc_tiles(w.R) : 0;
  SideStream* ss = nullptr;
  if (defer_wgrad && (ss = side_stream(s)) == nullptr) { set_error("%s: cannot create the side stream", fn); return NRM_ECUDA; }
  {
    KernelTimer t("head_backward", s);
    NRM_TRY(head_dgrad(params, w, precision, dlogits, grads, s));
    if (defer_wgrad) { ss->head_wgrad_pending = true; ss->wg_params = params; ss->wg_grads = grads; ss->wg_tiles = tiles; ss->wg_precision = tc ? precision : 0; }
    else NRM_TRY(launch_head_backward_wgrad(params, w, grads, s, tiles, tc ? precision : 0));
  }
  if (bn_bwd_sums != nullptr && bn_bwd_sums != w.bn_bwd_sums)
    NRM_CUDA(cudaMemcpyAsync(bn_bwd_sums, w.bn_bwd_sums, sizeof(double) * 2 * E, cudaMemcpyDeviceToDevice, s));
  return NRM_OK;
}

extern "C" int nrm_backward_head(int B, int H, int C, const float* params, int precision, const float* dlogits, float* grads,
                                 double* bn_bwd_sums, void* workspace, size_t workspace_bytes, void* stream) {
  return backward_head("nrm_backward_head", false, B, H, C, params, precision, dlogits, grads, bn_bwd_sums, workspace, workspace_bytes, stream);
}

extern "C" int nrm_backward_head_deferred(int B, int H, int C, const float* params, int precision, const float* dlogits, float* grads,
                                          double* bn_bwd_sums, void* workspace, size_t workspace_bytes, void* stream) {
  return backward_head("nrm_backward_head_deferred", true, B, H, C, params, precision, dlogits, grads, bn_bwd_sums, workspace, workspace_bytes, stream);
}

static int backward_encoder_impl(const char* fn, const BatchPtrs& in, int B, int H, int C, const float* params, int mode, int precision,
                                 const double* bn_bwd_sums, long long bn_global_rows, float* grads, void* workspace, size_t workspace_bytes,
                                 void* stream) {
  const int training = mode & NRM_MODE_BN_BATCH_STATS;
  Workspace w;
  NRM_TRY(get_workspace(fn, w, workspace, workspace_bytes, B, H, C, NRM_MODE_KEEP_FOR_BWD));
  cudaStream_t s = (cudaStream_t)stream;
  const double* sums = bn_bwd_sums ? bn_bwd_sums : w.bn_bwd_sums;
  const long long rows = bn_global_rows > 0 ? bn_global_rows : w.R;
  NRM_TRY(launch_bn_backward_combine(params, w, training, sums, rows, precision != NRM_PRECISION_FP32, s));
  return encoder_backward(in, params, w, precision, grads, s);   // also enqueues and joins the weight gradients nrm_backward_head_deferred left
}

extern "C" int nrm_backward_encoder(const double* x_history, const double* x_target, long long xt_bs,
                                    const double* x_global, long long xg_bs, int B, int H, int C, const float* params,
                                    int mode, int precision, const double* bn_bwd_sums, long long bn_global_rows,
                                    float* grads, void* workspace, size_t workspace_bytes, void* stream) {
  const char* fn = "nrm_backward_encoder";
  NRM_TRY(check_shape(fn, B, H, C));
  BatchPtrs in;
  NRM_TRY(packed_batch(fn, x_history, x_target, xt_bs, x_global, xg_bs, C, in));
  if (!params || !grads) { set_error("%s: null pointer", fn); return NRM_EINVAL; }
  return backward_encoder_impl(fn, in, B, H, C, params, mode, precision, bn_bwd_sums, bn_global_rows, grads, workspace, workspace_bytes, stream);
}

extern "C" int nrm_backward_encoder_compact(const nrm_compact_batch* batch, int B, int H, int C, const float* params, int mode, int precision,
                                            const double* bn_bwd_sums, long long bn_global_rows, float* grads, void* workspace,
                                            size_t workspace_bytes, void* stream) {
  const char* fn = "nrm_backward_encoder_compact";
  NRM_TRY(check_shape(fn, B, H, C));
  if (!params || !grads) { set_error("%s: null pointer", fn); return NRM_EINVAL; }
  BatchPtrs in;
  NRM_TRY(compact_batch(fn, batch, C, in));
  return backward_encoder_impl(fn, in, B, H, C, params, mode, precision, bn_bwd_sums, bn_global_rows, grads, workspace, workspace_bytes, stream);
}

extern "C" int nrm_backward(const double* x_history, const double* x_target, long long xt_bs, const double* x_global,
                            long long xg_bs, int B, int H, int C, const float* params, int mode, int precision,
                            const float* dlogits, float* grads, void* workspace, size_t workspace_bytes, void* stream) {
  const char* fn = "nrm_backward";
  NRM_TRY(check_shape(fn, B, H, C));
  BatchPtrs in;
  NRM_TRY(packed_batch(fn, x_history, x_target, xt_bs, x_global, xg_bs, C, in));
  NRM_TRY(backward_head(fn, true, B, H, C, params, precision, dlogits, grads, nullptr, workspace, workspace_bytes, stream));
  return backward_encoder_impl(fn, in, B, H, C, params, mode, precision, nullptr, 0, grads, workspace, workspace_bytes, stream);
}

extern "C" int nrm_backward_compact(const nrm_compact_batch* batch, int B, int H, int C, const float* params, int mode, int precision,
                                    const float* dlogits, float* grads, void* workspace, size_t workspace_bytes, void* stream) {
  const char* fn = "nrm_backward_compact";
  NRM_TRY(check_shape(fn, B, H, C));
  BatchPtrs in;
  NRM_TRY(compact_batch(fn, batch, C, in));
  NRM_TRY(backward_head(fn, true, B, H, C, params, precision, dlogits, grads, nullptr, workspace, workspace_bytes, stream));
  return backward_encoder_impl(fn, in, B, H, C, params, mode, precision, nullptr, 0, grads, workspace, workspace_bytes, stream);
}
