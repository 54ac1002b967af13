// fa_api.cu — the C ABI (include/fa_b200.h): validation, dispatch, host helpers.
// No TensorFlow / PyTorch / CuTe types cross this boundary.
#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <mutex>
#include <vector>

#include "../../include/fa_b200.h"
#include "fa_launch.h"
#include "sm100_tiles.cuh"

namespace fa {
// process-wide (autograd runs the backward on another thread than the forward)
static std::atomic<int64_t> g_launches{0};
static thread_local int g_last_cuda = 0;
static std::atomic<int> g_last_path{0};
static std::atomic<int> g_path_override{0};
static std::atomic<int> g_grad_precision{0};
void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }

// ---- optional per-kernel timing ------------------------------------------------------------
struct TimedLaunch { const char* name; cudaEvent_t start, stop; };
static std::atomic<int> g_timing{0};
static std::mutex g_timing_mu;
static std::vector<TimedLaunch> g_timed;

ScopedKernel::ScopedKernel(const char* name, cudaStream_t stream) : stream_(stream), slot_(-1) {
  count_launch();
  if (!g_timing.load(std::memory_order_relaxed)) return;
  TimedLaunch t{name, nullptr, nullptr};
  if (cudaEventCreate(&t.start) != cudaSuccess || cudaEventCreate(&t.stop) != cudaSuccess) return;
  cudaEventRecord(t.start, stream);
  std::lock_guard<std::mutex> g(g_timing_mu);
  slot_ = int(g_timed.size());
  g_timed.push_back(t);
}
ScopedKernel::~ScopedKernel() {
  if (slot_ < 0) return;
  std::lock_guard<std::mutex> g(g_timing_mu);
  // fa_kernel_timings() on another thread may have drained the list since the constructor ran
  if (size_t(slot_) < g_timed.size() && g_timed[slot_].stop) cudaEventRecord(g_timed[slot_].stop, stream_);
}
}  // namespace fa

namespace {

int make_rule(const fa_problem_t* p, FaRule* r) {
  if (!p) return FA_EINVAL_NULL;
  if (p->dtype < FA_F16 || p->dtype > FA_BF16) return FA_EINVAL_DTYPE;
  if (p->seq_dims != 1 && p->seq_dims != 2) return FA_EINVAL_SEQ_DIMS;
  if (p->d < 1 || p->v_d < 1 || p->batch < 0) return FA_EINVAL_SHAPE;
  return fa_make_rule(p->seq_dims, p->rule, p->window_size, p->log2_stride_size, p->is_causal,
                      p->sync_mode, p->q_shape, p->k_shape, p->q_index_base, p->k_index_base,
                      p->q_full_len, p->k_full_len, r);
}

// fp16 and bf16 share the tcgen05 16-bit family and every size rule
bool is16(int dtype) { return dtype == FA_F16 || dtype == FA_BF16; }
size_t elt(int dtype) { return is16(dtype) ? 2 : dtype == FA_F32 ? 4 : 8; }
size_t l_elt(int dtype) { return dtype == FA_F64 ? 8 : 4; }

int cuda_fail(cudaError_t e) {
  fa::g_last_cuda = int(e);
  return FA_ECUDA;
}

int fill_args(const fa_problem_t* p, fa::LaunchArgs* a) {
  int rc = make_rule(p, &a->rule);
  if (rc) return rc;
  a->dtype = p->dtype;
  a->d = p->d;
  a->v_d = p->v_d;
  a->batch = p->batch;
  a->accumulate = p->accumulate;
  if (p->layout != FA_LAYOUT_CHANNEL_FIRST && p->layout != FA_LAYOUT_CHANNEL_LAST) return FA_EINVAL_LAYOUT;
  if (p->layout == FA_LAYOUT_CHANNEL_LAST && (p->heads < 1 || p->batch % p->heads)) return FA_EINVAL_LAYOUT;
  a->layout = p->layout;
  a->heads = p->layout == FA_LAYOUT_CHANNEL_LAST ? p->heads : 0;
  a->grad_split = fa::g_grad_precision;
  // a key shard of a longer sequence (K/V ring): rows do not see all of their keys in this call
  a->partial_keys = (p->k_index_base != 0 || (p->k_full_len != 0 && p->k_full_len != a->rule.k.total)) ? 1 : 0;
  return 0;
}

}  // namespace

extern "C" {

const char* fa_version(void) { return "tf_flash_attention_b200 0.2 (sm_100a)"; }

const char* fa_strerror(int s) {
  switch (s) {
    case FA_OK: return "ok";
    case FA_EINVAL_NULL: return "null argument";
    case FA_EINVAL_DTYPE: return "unsupported dtype (expected float16, float32, float64 or bfloat16)";
    case FA_EINVAL_SEQ_DIMS: return "sequence dims must be 1 or 2";
    case FA_EINVAL_RULE: return "unknown masking rule";
    case FA_EINVAL_SYNC_MODE: return "Unsupported sync_mode";
    case FA_EINVAL_WINDOW: return "window_size must be >= 1";
    case FA_EINVAL_STRIDE:
      return "stride size is too big; please make sure the stride size/window size is within the range "
             "representable by int32_t";
    case FA_EINVAL_SHAPE: return "invalid or unsupported shape";
    case FA_EINVAL_WORKSPACE: return "workspace too small";
    case FA_EINVAL_RANK: return "The number of dimensions of the inputs is inconsistent or too small";
    case FA_EINVAL_CHANNEL: return "The channel dimensions should be equal";
    case FA_EINVAL_BATCH: return "The batch shape of all inputs should be equal";
    case FA_EINVAL_SEQ_SHAPE: return "The sequence shapes are inconsistent";
    case FA_EINVAL_LAYOUT:
      return "channel-last operands are read directly only by the 16-bit tensor-core kernels (channels multiples of 8 up "
             "to 128, 16-byte-aligned tensors, heads >= 1 dividing batch); use fa_layout_transpose otherwise";
    case FA_ECUDA: return "CUDA error (see fa_last_cuda_error)";
    case FA_ENODEVICE: return "no sm_100 CUDA device is current";
    default: return "unknown status";
  }
}

int fa_last_cuda_error(void) { return fa::g_last_cuda; }
int fa_last_path(void) { return fa::g_last_path; }
int64_t fa_launch_count(int reset) {
  return reset ? fa::g_launches.exchange(0) : fa::g_launches.load();
}
void fa_set_path_override(int path) { fa::g_path_override = path; }
int fa_set_grad_precision(int mode) {
  if (mode < 0 || mode > 2) return FA_EINVAL_SHAPE;
  fa::g_grad_precision = mode;
  return FA_OK;
}

void fa_kernel_timing(int enable) { fa::g_timing.store(enable ? 1 : 0); }

int fa_kernel_timings(int max_entries, const char** names, float* ms) {
  std::lock_guard<std::mutex> g(fa::g_timing_mu);
  int n = 0;
  for (auto& t : fa::g_timed) {
    float v = -1.f;
    if (cudaEventSynchronize(t.stop) == cudaSuccess) cudaEventElapsedTime(&v, t.start, t.stop);
    if (n < max_entries) {
      if (names) names[n] = t.name;
      if (ms) ms[n] = v;
      ++n;
    }
    cudaEventDestroy(t.start);
    cudaEventDestroy(t.stop);
  }
  fa::g_timed.clear();
  return n;
}

size_t fa_workspace_bytes(const fa_problem_t* p, int is_backward) {
  fa::LaunchArgs a{};
  if (fill_args(p, &a)) return 0;
  size_t g = fa::generic_workspace_bytes(p->dtype, p->batch, a.rule.q.total, is_backward != 0);
  size_t s = 0;
  a.variant = fa::g_path_override;
  if (is16(p->dtype)) s = fa::sm100_f16_workspace_bytes(a, is_backward != 0);
  if (p->dtype == FA_F32 && is_backward && fa::g_path_override != 1) {
    fa::LaunchArgs probe = a;
    probe.workspace = reinterpret_cast<void*>(uintptr_t(256));   // a probe: only shape / size rules are evaluated
    probe.workspace_bytes = ~size_t(0);
    if (fa::sm100_f32_backward_supports(probe)) s = fa::sm100_f32_backward_workspace_bytes(a);
  }
  if (p->dtype == FA_F32 && !is_backward) {
    // hi / lo TF32 copies of Q, K, V (and a padded O) for the 3xTF32 forward, when that kernel takes the shape
    fa::LaunchArgs probe = a;
    probe.o = nullptr;
    probe.workspace = reinterpret_cast<void*>(uintptr_t(256));
    probe.workspace_bytes = ~size_t(0);
    if (fa::g_path_override != 1 && fa::sm100_f32_forward_supports(probe)) s = fa::sm100_f32_forward_workspace_bytes(a);
  }
  return g > s ? g : s;
}

int fa_forward(const fa_problem_t* p, const void* q, const void* k, const void* v, void* o, void* l,
               void* m, void* workspace, size_t workspace_bytes, void* stream) {
  fa::LaunchArgs a{};
  int rc = fill_args(p, &a);
  if (rc) return rc;
  if (p->batch == 0) return FA_OK;
  if (!q || !k || !v || !o || !l || !m) return FA_EINVAL_NULL;
  const size_t need = fa_workspace_bytes(p, 0);
  if (workspace_bytes < need || (!workspace && need)) return FA_EINVAL_WORKSPACE;
  a.q = q; a.k = k; a.v = v; a.o = o; a.l = l; a.m = m;
  a.workspace = workspace; a.workspace_bytes = workspace_bytes;
  a.variant = fa::g_path_override;
  cudaStream_t st = (cudaStream_t)stream;
  cudaError_t e;
  if (fa::g_path_override != 1 && is16(p->dtype) && fa::sm100_f16_forward_supports(a)) {
    fa::g_last_path = 2;
    e = fa::sm100_f16_forward(a, st);
  } else if (fa::g_path_override != 1 && p->dtype == FA_F32 && fa::sm100_f32_forward_supports(a)) {
    fa::g_last_path = 3;
    e = fa::sm100_f32_forward(a, st);
  } else if (fa::g_path_override != 1 && p->dtype == FA_F64 && fa::f64_dmma_forward_supports(a)) {
    fa::g_last_path = 4;
    e = fa::f64_dmma_forward(a, st);
  } else {
    if (a.layout != 0) return FA_EINVAL_LAYOUT;
    if (!fa::generic_supports(a, false)) return FA_EINVAL_SHAPE;
    fa::g_last_path = 1;
    e = fa::generic_forward(a, st);
  }
  return e == cudaSuccess ? FA_OK : cuda_fail(e);
}

int fa_backward(const fa_problem_t* p, const void* q, const void* k, const void* v, const void* o,
                const void* l, const void* m, const void* d_o, void* d_q, void* d_k, void* d_v,
                void* workspace, size_t workspace_bytes, void* stream) {
  fa::LaunchArgs a{};
  int rc = fill_args(p, &a);
  if (rc) return rc;
  if (p->batch == 0) return FA_OK;
  if (!q || !k || !v || !o || !l || !m || !d_o || !d_q || !d_k || !d_v) return FA_EINVAL_NULL;
  const size_t need = fa_workspace_bytes(p, 1);
  if (workspace_bytes < need || (!workspace && need)) return FA_EINVAL_WORKSPACE;
  a.q = q; a.k = k; a.v = v; a.o = (void*)o; a.l = (void*)l; a.m = (void*)m; a.d_o = d_o;
  a.d_q = d_q; a.d_k = d_k; a.d_v = d_v;
  a.workspace = workspace; a.workspace_bytes = workspace_bytes;
  a.variant = fa::g_path_override;
  cudaStream_t st = (cudaStream_t)stream;
  cudaError_t e;
  if (fa::g_path_override != 1 && is16(p->dtype) && fa::sm100_f16_backward_supports(a)) {
    fa::g_last_path = 2;
    e = fa::sm100_f16_backward(a, st);
  } else if (fa::g_path_override != 1 && p->dtype == FA_F32 && fa::sm100_f32_backward_supports(a)) {
    fa::g_last_path = 3;
    e = fa::sm100_f32_backward(a, st);
  } else if (fa::g_path_override != 1 && p->dtype == FA_F64 && fa::f64_dmma_backward_supports(a)) {
    fa::g_last_path = 4;
    e = fa::f64_dmma_backward(a, st);
  } else {
    if (a.layout != 0) return FA_EINVAL_LAYOUT;
    if (!fa::generic_supports(a, true)) return FA_EINVAL_SHAPE;
    fa::g_last_path = 1;
    e = fa::generic_backward(a, st);
  }
  return e == cudaSuccess ? FA_OK : cuda_fail(e);
}

// dQ ADDED into an fp32 accumulator inside the backward launch (K/V ring: every block's dQ used to go through the fused
// kernel's scratch, a convert pass, an fp16 tensor and fa_grad_accumulate; the kernel's reduce-add can land in the
// accumulator directly).
static int fill_accumulate_args(const fa_problem_t* p, const void* q, const void* k, const void* v, const void* o,
                                const void* l, const void* m, const void* d_o, void* dq_acc, void* d_k, void* d_v,
                                int64_t dq_fold, void* workspace, size_t workspace_bytes, fa::LaunchArgs* a) {
  int rc = fill_args(p, a);
  if (rc) return rc;
  a->q = q; a->k = k; a->v = v; a->o = (void*)o; a->l = (void*)l; a->m = (void*)m; a->d_o = d_o;
  a->d_q = dq_acc; a->d_k = d_k; a->d_v = d_v;
  a->workspace = workspace; a->workspace_bytes = workspace_bytes;
  a->variant = fa::g_path_override;
  a->grad_acc = 1;
  a->dq_fold = dq_fold > 0 ? dq_fold : p->batch;
  return 0;
}

int fa_backward_accumulate_supported(const fa_problem_t* p, int64_t dq_fold) {
  fa::LaunchArgs a{};
  void* dummy = reinterpret_cast<void*>(uintptr_t(256));   // a probe: only shape rules are evaluated
  if (!p || fill_accumulate_args(p, dummy, dummy, dummy, dummy, dummy, dummy, dummy, dummy, dummy, dummy, dq_fold, dummy,
                                 ~size_t(0), &a))
    return 0;
  return (is16(p->dtype) && fa::g_path_override != 1 && p->batch > 0 && fa::sm100_f16_backward_accumulate_supports(a)) ? 1 : 0;
}

int fa_backward_accumulate(const fa_problem_t* p, const void* q, const void* k, const void* v, const void* o,
                           const void* l, const void* m, const void* d_o, void* dq_acc, void* d_k, void* d_v,
                           int64_t dq_fold, void* workspace, size_t workspace_bytes, void* stream) {
  if (!p) return FA_EINVAL_NULL;
  fa::LaunchArgs a{};
  int rc = fill_accumulate_args(p, q, k, v, o, l, m, d_o, dq_acc, d_k, d_v, dq_fold, workspace, workspace_bytes, &a);
  if (rc) return rc;
  if (p->batch == 0) return FA_OK;
  if (!q || !k || !v || !o || !l || !m || !d_o || !dq_acc || !d_k || !d_v) return FA_EINVAL_NULL;
  const size_t need = fa_workspace_bytes(p, 1);
  if (workspace_bytes < need || (!workspace && need)) return FA_EINVAL_WORKSPACE;
  if (!is16(p->dtype) || fa::g_path_override == 1 || !fa::sm100_f16_backward_accumulate_supports(a))
    return FA_EINVAL_SHAPE;   // callers fall back to fa_backward + fa_grad_accumulate
  fa::g_last_path = 2;
  cudaError_t e = fa::sm100_f16_backward(a, (cudaStream_t)stream);
  return e == cudaSuccess ? FA_OK : cuda_fail(e);
}

// Which kernel family a call will take, and when it is the generic one, why (host only). The tensor-core families
// decline a problem silently (fa_last_path() afterwards is the only trace); a framework can ask beforehand.
int fa_dispatch_path(const fa_problem_t* p, int is_backward, char* reason, size_t reason_len) {
  auto say = [&](const char* msg) {
    if (reason && reason_len) snprintf(reason, reason_len, "%s", msg);
  };
  say("");
  if (!p) return FA_EINVAL_NULL;
  fa::LaunchArgs a{};
  int rc = fill_args(p, &a);
  if (rc) return rc;
  void* al = reinterpret_cast<void*>(uintptr_t(256));   // probe: aligned tensors, workspace as large as asked for
  a.q = a.k = a.v = a.d_o = al;
  a.o = a.l = a.m = a.d_q = a.d_k = a.d_v = a.workspace = al;
  a.workspace_bytes = ~size_t(0);
  a.variant = fa::g_path_override;
  const bool bwd = is_backward != 0;
  if (fa::g_path_override == 1) {
    say("fa_set_path_override(1): generic kernels forced");
    return a.layout ? FA_EINVAL_LAYOUT : fa::generic_supports(a, bwd) ? 1 : FA_EINVAL_SHAPE;
  }
  const int64_t nq = a.rule.q.total, nk = a.rule.k.total;
  const int64_t cap = 32 * int64_t(fa::sm100::kMaxTileWords);   // streamed tiles of a CTA's schedule
  if (is16(p->dtype) && (bwd ? fa::sm100_f16_backward_supports(a) : fa::sm100_f16_forward_supports(a))) return 2;
  if (p->dtype == FA_F32 && (bwd ? fa::sm100_f32_backward_supports(a) : fa::sm100_f32_forward_supports(a))) return 3;
  if (p->dtype == FA_F64 && (bwd ? fa::f64_dmma_backward_supports(a) : fa::f64_dmma_forward_supports(a))) return 4;
  const int max_ch = is16(p->dtype) ? 128 : 64;
  const int64_t tile = (is16(p->dtype) && !bwd && (p->d > 64 || p->v_d > 64)) ? 128 : 64;
  if (a.layout != 0) {
    say("channel-last operands are read directly only by the 16-bit tensor-core kernels (channels multiples of 8 up to "
        "128)");
    return FA_EINVAL_LAYOUT;
  }
  if (p->d > 256 || p->v_d > 256) {
    if (!fa::generic_supports(a, bwd)) {
      say("more than 256 channels: batch x tiles x channel slices exceeds a 31-bit grid");
      return FA_EINVAL_SHAPE;
    }
    say("more than 256 channels: channel-sliced generic kernels (each CTA owns at most 256 output channels and "
        "recomputes S for them)");
    return 1;
  }
  if (p->d > max_ch || p->v_d > max_ch)
    say(is16(p->dtype) ? "more than 128 channels: generic kernels" : "more than 64 channels: generic kernels");
  else if (!bwd && a.accumulate)
    say("accumulate = 1 is served by the generic forward kernels");
  else if (p->dtype != FA_F64 && ((nk + tile - 1) / tile > cap || (bwd && (nq + 63) / 64 > cap)))
    say("sequence longer than the 2048 streamed tiles a CTA's schedule holds (131072 positions at 64 per tile, 262144 "
        "keys for the head_dim-128 forward): generic kernels; shard the sequence (K/V ring) to stay on the tensor cores");
  else
    say("batch x tiles exceeds a 31-bit grid: generic kernels");
  return 1;
}

// ---- layout adapter ------------------------------------------------------------------------------
int fa_layout_transpose(int32_t dtype, const void* x, void* y, int64_t batch, int64_t seq, int32_t heads,
                        int32_t channels, int to_channel_first, void* stream) {
  if (dtype < FA_F16 || dtype > FA_BF16) return FA_EINVAL_DTYPE;
  if (batch < 0 || seq < 0 || heads < 0 || channels < 0) return FA_EINVAL_SHAPE;
  if (batch * heads > 0x7fffffffLL || (seq + 31) / 32 > 65535 || (channels + 31) / 32 > 65535) return FA_EINVAL_SHAPE;
  if (batch * seq * heads * channels == 0) return FA_OK;
  if (!x || !y) return FA_EINVAL_NULL;
  cudaError_t e = fa::layout_transpose(dtype, x, y, batch, seq, heads, channels, to_channel_first, fa::g_path_override, (cudaStream_t)stream);
  return e == cudaSuccess ? FA_OK : cuda_fail(e);
}

// ---- gradient shards (ring backward) ---------------------------------------------------------
int fa_grad_accumulate(int32_t dtype, const void* part, void* acc, int64_t n, int first, void* stream) {
  if (dtype < FA_F16 || dtype > FA_BF16) return FA_EINVAL_DTYPE;
  if (n < 0) return FA_EINVAL_SHAPE;
  if (n == 0) return FA_OK;
  if (!part || !acc) return FA_EINVAL_NULL;
  cudaError_t e = fa::grad_accumulate(dtype, part, acc, n, first, (cudaStream_t)stream);
  return e == cudaSuccess ? FA_OK : cuda_fail(e);
}
int fa_grad_finalize(int32_t dtype, const void* acc, void* out, int64_t n, void* stream) {
  if (dtype < FA_F16 || dtype > FA_BF16) return FA_EINVAL_DTYPE;
  if (n < 0) return FA_EINVAL_SHAPE;
  if (n == 0) return FA_OK;
  if (!acc || !out) return FA_EINVAL_NULL;
  cudaError_t e = fa::grad_finalize(dtype, acc, out, n, (cudaStream_t)stream);
  return e == cudaSuccess ? FA_OK : cuda_fail(e);
}

// ---- partial results over key shards (K/V ring) -------------------------------------------------
int fa_partial_merge(const fa_problem_t* p, const void* o_part, const void* l_part, const void* m_part,
                     void* o_acc, void* l_acc, void* m_acc, int first, void* stream) {
  fa::LaunchArgs a{};
  int rc = fill_args(p, &a);
  if (rc) return rc;
  if (a.layout != 0) return FA_EINVAL_LAYOUT;
  if (p->batch == 0) return FA_OK;
  if (!o_part || !l_part || !m_part || !o_acc || !l_acc || !m_acc) return FA_EINVAL_NULL;
  cudaError_t e = fa::partial_merge(a, o_part, l_part, m_part, o_acc, l_acc, m_acc, first, (cudaStream_t)stream);
  return e == cudaSuccess ? FA_OK : cuda_fail(e);
}

int fa_partial_finalize(const fa_problem_t* p, const void* o_acc, const void* l_acc, const void* m_acc, void* o,
                        void* l, void* m, void* stream) {
  fa::LaunchArgs a{};
  int rc = fill_args(p, &a);
  if (rc) return rc;
  if (a.layout != 0) return FA_EINVAL_LAYOUT;
  if (p->batch == 0) return FA_OK;
  if (!o_acc || !l_acc || !m_acc || !o || !l || !m) return FA_EINVAL_NULL;
  cudaError_t e = fa::partial_finalize(a, o_acc, l_acc, m_acc, o, l, m, (cudaStream_t)stream);
  return e == cudaSuccess ? FA_OK : cuda_fail(e);
}

// ---- host helpers on the shared rule code ---------------------------------------------------

int fa_count_attended(const fa_problem_t* p, int64_t* nnz) {
  FaRule r;
  int rc = make_rule(p, &r);
  if (rc) return rc;
  if (!nnz) return FA_EINVAL_NULL;
  int64_t total = 0;
  if (r.rule == 0) {
    total = int64_t(r.q.total) * r.k.total;
  } else {
    // per-row: walk only the K tiles the schedule keeps, count FULL tiles wholesale
    const int TK = 128;
    std::vector<FaPos> kpos(r.k.total);
    for (int32_t j = 0; j < r.k.total; ++j) kpos[j] = fa_pos(r, r.k, j);
    for (int32_t i = 0; i < r.q.total; ++i) {
      FaPos qp = fa_pos(r, r.q, i);
      int32_t f, l;
      fa_k_tile_range(r, i, i, TK, &f, &l);
      for (int32_t t = f; t <= l; ++t) {
        int32_t k0 = t * TK, k1 = std::min(k0 + TK, r.k.total) - 1;
        int cls = fa_classify(r, i, i, k0, k1);
        if (cls == FA_TILE_SKIP) continue;
        if (cls == FA_TILE_FULL) {
          total += k1 - k0 + 1;
          continue;
        }
        for (int32_t j = k0; j <= k1; ++j) total += fa_attend(r, qp, kpos[j]) ? 1 : 0;
      }
    }
  }
  *nnz = total;
  return FA_OK;
}

int fa_pattern_mask(const fa_problem_t* p, uint8_t* mask) {
  FaRule r;
  int rc = make_rule(p, &r);
  if (rc) return rc;
  if (!mask) return FA_EINVAL_NULL;
  std::vector<FaPos> kpos(r.k.total);
  for (int32_t j = 0; j < r.k.total; ++j) kpos[j] = fa_pos(r, r.k, j);
  for (int32_t i = 0; i < r.q.total; ++i) {
    FaPos qp = fa_pos(r, r.q, i);
    uint8_t* row = mask + int64_t(i) * r.k.total;
    for (int32_t j = 0; j < r.k.total; ++j) row[j] = fa_attend(r, qp, kpos[j]) ? 1 : 0;
  }
  return FA_OK;
}

// Same pattern as fa_pattern_mask but assembled from the closed-form 32-column masks the tcgen05
// kernels use (fa_fast_mask32), both with queries resident (forward / dQ kernels) and with keys resident
// (dK/dV kernel), tiles of `tile` streamed entries. Returns FA_EINVAL_RULE for rules that have no closed
// form (local with log2_stride > 0 uses the element rule in the kernels as well).
int fa_pattern_mask_fast(const fa_problem_t* p, int32_t tile, int32_t resident_is_q, uint8_t* mask) {
  FaRule r;
  int rc = make_rule(p, &r);
  if (rc) return rc;
  if (!mask || tile < 32 || tile % 32) return FA_EINVAL_NULL;
  const FaSeqMap& res_map = resident_is_q ? r.q : r.k;
  const FaSeqMap& str_map = resident_is_q ? r.k : r.q;
  for (int32_t i = 0; i < res_map.total; ++i) {
    const FaPos rp = fa_pos(r, res_map, i);
    for (int32_t s0 = 0; s0 < str_map.total; s0 += tile) {
      const int32_t nvalid = std::min(tile, str_map.total - s0);
      for (int32_t c0 = 0; c0 < tile; c0 += 32) {
        const uint32_t bits = fa_fast_mask32(r, resident_is_q != 0, rp, s0, c0, nvalid);
        for (int e = 0; e < 32; ++e) {
          const int32_t j = s0 + c0 + e;
          if (j >= str_map.total) {
            if ((bits >> e) & 1u) return FA_EINVAL_SHAPE;  // a bit outside the sequence: bug
            continue;
          }
          const int64_t idx = resident_is_q ? int64_t(i) * r.k.total + j : int64_t(j) * r.k.total + i;
          mask[idx] = (bits >> e) & 1u;
        }
      }
    }
  }
  return FA_OK;
}

int fa_orders(const fa_problem_t* p, int32_t* q_order, int32_t* k_order, int32_t* ref_shape) {
  FaRule r;
  int rc = make_rule(p, &r);
  if (rc) return rc;
  if (q_order)
    for (int32_t i = 0; i < r.q.total; ++i) q_order[i] = fa_pos(r, r.q, i).order;
  if (k_order)
    for (int32_t j = 0; j < r.k.total; ++j) k_order[j] = fa_pos(r, r.k, j).order;
  if (ref_shape) {
    ref_shape[0] = r.ref0;
    if (r.dims == 2) ref_shape[1] = r.ref1;
  }
  return FA_OK;
}

int fa_classify_tiles(const fa_problem_t* p, int32_t tile_q, int32_t tile_k, uint8_t* cls) {
  FaRule r;
  int rc = make_rule(p, &r);
  if (rc) return rc;
  if (!cls || tile_q < 1 || tile_k < 1) return FA_EINVAL_NULL;
  const int32_t nqt = (r.q.total + tile_q - 1) / tile_q, nkt = (r.k.total + tile_k - 1) / tile_k;
  for (int32_t a = 0; a < nqt; ++a) {
    int32_t q0 = a * tile_q, q1 = std::min(q0 + tile_q, r.q.total) - 1;
    int32_t f, l;
    fa_k_tile_range(r, q0, q1, tile_k, &f, &l);
    for (int32_t b = 0; b < nkt; ++b) {
      int32_t k0 = b * tile_k, k1 = std::min(k0 + tile_k, r.k.total) - 1;
      int c = (b < f || b > l) ? FA_TILE_SKIP : fa_classify(r, q0, q1, k0, k1);
      // the dK/dV kernels walk the transposed range; a tile either range drops is reported as
      // SKIP so that the tests can verify both ranges only ever drop empty tiles
      int32_t qf, ql;
      fa_q_tile_range(r, k0, k1, tile_q, &qf, &ql);
      if (a < qf || a > ql) c = FA_TILE_SKIP;
      cls[int64_t(a) * nkt + b] = uint8_t(c);
    }
  }
  return FA_OK;
}

// ---- the reference's FLOPs estimate ---------------------------------------------------------
// Restates FlashAttentionLauncher::EstimateForwardFlops (flash_attention.cu:2069-2144) with the
// reference's own tile configuration (flash_attention.cu:1977-2012, flash_attention.h:187-204) and
// its own IsSkipped predicates (flash_attention.h:48-115), including their quirks, so that the
// number TF's profiler shows stays comparable. Note the reference does not multiply by batch.
namespace {
struct RefCoords { int32_t c[2]; };
inline int32_t ilog2(int32_t n) { int32_t l = 0; while ((int64_t(1) << (l + 1)) <= n) ++l; return l; }
RefCoords ref_coords(const FaRule& r, int32_t order) {
  RefCoords o;
  o.c[0] = order & (r.ref0 - 1);
  o.c[1] = r.dims == 2 ? (order >> r.ref_log2_0) & (r.ref1 - 1) : 0;
  return o;
}
int32_t ref_order(const FaRule& r, const RefCoords& c) {
  return c.c[0] + (r.dims == 2 ? (c.c[1] << r.ref_log2_0) : 0);
}
bool ref_is_skipped(const FaRule& r, int32_t minQ, int32_t maxQ, int32_t minK, int32_t maxK) {
  if (r.rule == 0) return false;
  if (r.rule == 1) return maxQ < minK;
  const int32_t sw = r.window << r.log2_stride;
  const int32_t look = r.causal ? 1 : sw;
  RefCoords a = ref_coords(r, minQ), b = ref_coords(r, maxQ), lo, hi;
  const int32_t lim[2] = {r.ref0, r.ref1};
  for (int i = 0; i < 2; ++i) {
    lo.c[i] = std::max(a.c[i] - sw + 1, 0);
    hi.c[i] = std::min(b.c[i] + look, lim[i]) - 1;
  }
  return maxK < ref_order(r, lo) || minK > ref_order(r, hi);
}
}  // namespace

int fa_estimate_forward_flops(const fa_problem_t* p, int32_t shared_mem_bytes, float* flops) {
  FaRule r;
  int rc = make_rule(p, &r);
  if (rc) return rc;
  if (!flops) return FA_EINVAL_NULL;
  const int32_t smem = shared_mem_bytes > 0 ? shared_mem_bytes : 232448;
  const int32_t sz = int32_t(elt(p->dtype));
  const int32_t Br = std::max(32, 128 / sz);
  const int32_t pad = sz == 2 ? 2 : 1;
  const int32_t d = p->d, v_d = p->v_d, q = r.q.total, k = r.k.total;
  const int32_t Bc = (smem - Br * (1 + 1 + d) * sz) / ((d + v_d + (Br + pad)) * sz);
  if (Bc <= 0) return FA_EINVAL_SHAPE;
  const int32_t nBr = (q + Br - 1) / Br, nBc = (k + Bc - 1) / Bc;
  const int32_t per_pair = Br * Bc * (2 * d - 1) + (Br * (Bc - 1) * 2 + Br * Bc * 2) + Br * 7 +
                           Br * (Bc + v_d) + Br * v_d * (2 * Bc - 1);
  const int32_t max_order = r.ref0 * r.ref1 - 1;
  float f = 0.0f;
  for (int32_t bc = 0; bc < nBc; ++bc) {
    const int32_t minK = fa_pos(r, r.k, bc * Bc).order;
    const int32_t maxK = std::min(fa_pos(r, r.k, (bc + 1) * Bc - 1).order, max_order);
    for (int32_t br = 0; br < nBr; ++br) {
      const int32_t minQ = fa_pos(r, r.q, br * Br).order;
      const int32_t maxQ = std::min(fa_pos(r, r.q, (br + 1) * Br - 1).order, max_order);
      if (ref_is_skipped(r, minQ, maxQ, minK, maxK)) continue;
      f += per_pair;
    }
  }
  *flops = f;
  return FA_OK;
}

// ---- shape validation as in the reference OpKernels -------------------------------------------
namespace {
struct Split { int64_t batch; int64_t ch; int32_t seq[2]; bool seq_ok; std::vector<int64_t> bdims; };
bool split(int32_t seq_dims, int32_t rank, const int64_t* dims, bool has_channel, Split* s) {
  const int lead = rank - seq_dims - (has_channel ? 1 : 0);
  if (lead < 0) return false;
  s->batch = 1;
  s->bdims.assign(dims, dims + lead);
  for (int i = 0; i < lead; ++i) s->batch *= dims[i];
  s->ch = has_channel ? dims[lead] : 0;
  s->seq_ok = true;
  s->seq[0] = s->seq[1] = 1;
  for (int i = 0; i < seq_dims; ++i) {
    int64_t v = dims[lead + (has_channel ? 1 : 0) + i];
    if (v < 1 || v > 0x7fffffffLL) s->seq_ok = false;
    s->seq[i] = int32_t(v);
  }
  return true;
}
}  // namespace

int fa_check_forward_shapes(int32_t seq_dims, int32_t rank_q, const int64_t* q_dims, int32_t rank_k,
                            const int64_t* k_dims, int32_t rank_v, const int64_t* v_dims,
                            fa_problem_t* p) {
  if (!p || !q_dims || !k_dims || !v_dims) return FA_EINVAL_NULL;
  if (seq_dims != 1 && seq_dims != 2) return FA_EINVAL_SEQ_DIMS;
  // "The number of dimensions of Q, K, and V should be equal" / ">= SequenceDims+2" (forward.cc:100-104)
  if (rank_q != rank_k || rank_k != rank_v) return FA_EINVAL_RANK;
  if (rank_q < seq_dims + 2) return FA_EINVAL_RANK;
  Split Q, K, V;
  split(seq_dims, rank_q, q_dims, true, &Q);
  split(seq_dims, rank_k, k_dims, true, &K);
  split(seq_dims, rank_v, v_dims, true, &V);
  if (Q.ch != K.ch) return FA_EINVAL_CHANNEL;                                    // forward.cc:126-127
  if (Q.bdims != K.bdims || Q.bdims != V.bdims) return FA_EINVAL_BATCH;          // forward.cc:129-130
  if (K.seq[0] != V.seq[0] || K.seq[1] != V.seq[1]) return FA_EINVAL_SEQ_SHAPE;  // forward.cc:132-133
  if (!Q.seq_ok || !K.seq_ok || Q.ch < 1 || V.ch < 1 || Q.ch > 0x7fffffffLL || V.ch > 0x7fffffffLL)
    return FA_EINVAL_SHAPE;
  p->seq_dims = seq_dims;
  p->batch = Q.batch;
  p->d = int32_t(Q.ch);
  p->v_d = int32_t(V.ch);
  for (int i = 0; i < 2; ++i) {
    p->q_shape[i] = i < seq_dims ? Q.seq[i] : 0;
    p->k_shape[i] = i < seq_dims ? K.seq[i] : 0;
  }
  return FA_OK;
}

int fa_check_backward_shapes(int32_t seq_dims, int32_t rank_q, const int64_t* q_dims, int32_t rank_k,
                             const int64_t* k_dims, int32_t rank_v, const int64_t* v_dims,
                             int32_t rank_o, const int64_t* o_dims, int32_t rank_l,
                             const int64_t* l_dims, int32_t rank_m, const int64_t* m_dims,
                             int32_t rank_do, const int64_t* do_dims, fa_problem_t* p) {
  if (!p || !q_dims || !k_dims || !v_dims || !o_dims || !l_dims || !m_dims || !do_dims)
    return FA_EINVAL_NULL;
  if (seq_dims != 1 && seq_dims != 2) return FA_EINVAL_SEQ_DIMS;
  // backward.cc:197-208
  if (!(rank_q == rank_k && rank_k == rank_v && rank_v == rank_o && rank_o == rank_do)) return FA_EINVAL_RANK;
  if (!(rank_l == rank_m && rank_m == rank_q - 1)) return FA_EINVAL_RANK;
  if (rank_q < seq_dims + 2) return FA_EINVAL_RANK;
  Split Q, K, V, O, L, M, DO;
  split(seq_dims, rank_q, q_dims, true, &Q);
  split(seq_dims, rank_k, k_dims, true, &K);
  split(seq_dims, rank_v, v_dims, true, &V);
  split(seq_dims, rank_o, o_dims, true, &O);
  split(seq_dims, rank_l, l_dims, false, &L);
  split(seq_dims, rank_m, m_dims, false, &M);
  split(seq_dims, rank_do, do_dims, true, &DO);
  if (Q.ch != K.ch) return FA_EINVAL_CHANNEL;  // backward.cc:243-244
  if (V.ch != O.ch) return FA_EINVAL_CHANNEL;  // backward.cc:245-246
  if (!(Q.bdims == K.bdims && Q.bdims == V.bdims && V.bdims == O.bdims && O.bdims == L.bdims &&
        L.bdims == M.bdims && M.bdims == DO.bdims))
    return FA_EINVAL_BATCH;  // backward.cc:249-252
  auto same = [](const Split& a, const Split& b) { return a.seq[0] == b.seq[0] && a.seq[1] == b.seq[1]; };
  if (!same(K, V)) return FA_EINVAL_SEQ_SHAPE;  // backward.cc:254-255
  if (!(same(Q, O) && same(O, L) && same(L, M) && same(M, DO))) return FA_EINVAL_SEQ_SHAPE;  // :257-258
  // the reference never checks dO's channel count against V's; a mismatch would read out of
  // bounds there, so it is rejected here.
  if (DO.ch != V.ch) return FA_EINVAL_CHANNEL;
  if (!Q.seq_ok || !K.seq_ok || Q.ch < 1 || V.ch < 1 || Q.ch > 0x7fffffffLL || V.ch > 0x7fffffffLL)
    return FA_EINVAL_SHAPE;
  p->seq_dims = seq_dims;
  p->batch = Q.batch;
  p->d = int32_t(Q.ch);
  p->v_d = int32_t(V.ch);
  for (int i = 0; i < 2; ++i) {
    p->q_shape[i] = i < seq_dims ? Q.seq[i] : 0;
    p->k_shape[i] = i < seq_dims ? K.seq[i] : 0;
  }
  return FA_OK;
}

// ---- host-buffer entry points (the e2e path) ----------------------------------------------------
namespace {
size_t align_up(size_t v) { return (v + 255) & ~size_t(255); }
struct Arena {
  size_t q, k, v, o, l, m, d_o, d_q, d_k, d_v, ws, total;
  size_t nq_b, nk_b, nv_b, no_b, nl_b, nm_b;
};
int arena_layout(const fa_problem_t* p, int bwd, Arena* a) {
  FaRule r;
  int rc = make_rule(p, &r);
  if (rc) return rc;
  // the host pipelines cut the batch into contiguous chunks: only the reference's channel-first layout is contiguous
  // per batch element
  if (p->layout != FA_LAYOUT_CHANNEL_FIRST) return FA_EINVAL_LAYOUT;
  const size_t e = elt(p->dtype), b = size_t(p->batch);
  a->nq_b = e * b * p->d * r.q.total;
  a->nk_b = e * b * p->d * r.k.total;
  a->nv_b = e * b * p->v_d * r.k.total;
  a->no_b = e * b * p->v_d * r.q.total;
  a->nl_b = l_elt(p->dtype) * b * r.q.total;
  a->nm_b = e * b * r.q.total;
  size_t off = 0;
  auto take = [&off](size_t n) { size_t o = off; off += align_up(n); return o; };
  a->q = take(a->nq_b); a->k = take(a->nk_b); a->v = take(a->nv_b);
  a->o = take(a->no_b); a->l = take(a->nl_b); a->m = take(a->nm_b);
  if (bwd) {
    a->d_o = take(a->no_b); a->d_q = take(a->nq_b); a->d_k = take(a->nk_b); a->d_v = take(a->nv_b);
  }
  a->ws = off;
  off += align_up(fa_workspace_bytes(p, bwd));
  a->total = off;
  return 0;
}
}  // namespace

size_t fa_host_arena_bytes(const fa_problem_t* p, int is_backward) {
  Arena a;
  if (arena_layout(p, is_backward, &a)) return 0;
  return a.total;
}

#define FA_CU(x)                                   \
  do {                                             \
    cudaError_t e_ = (x);                          \
    if (e_ != cudaSuccess) return cuda_fail(e_);   \
  } while (0)

namespace {
// Host-buffer calls are pipelined over chunks of the batch on three streams: upload of chunk c+1,
// compute of chunk c (on the caller's stream) and download of chunk c-1 overlap (PCIe is full duplex).
// One pipe (two copy streams + a growing pool of events) is kept per (device, caller stream) for the life of the
// process, so a host-buffer call creates nothing on the hot path.
struct HostPipe {
  cudaStream_t in = nullptr, out = nullptr;
  std::vector<cudaEvent_t> ev;
  std::mutex busy;   // one host-buffer call at a time per (device, stream)
  cudaError_t reserve(int n_events) {
    cudaError_t e;
    if (!in && (e = cudaStreamCreateWithFlags(&in, cudaStreamNonBlocking)) != cudaSuccess) return e;
    if (!out && (e = cudaStreamCreateWithFlags(&out, cudaStreamNonBlocking)) != cudaSuccess) return e;
    while (int(ev.size()) < n_events) {
      cudaEvent_t x = nullptr;
      if ((e = cudaEventCreateWithFlags(&x, cudaEventDisableTiming)) != cudaSuccess) return e;
      ev.push_back(x);
    }
    return cudaSuccess;
  }
};
std::mutex g_pipes_mu;
std::vector<std::pair<std::pair<int, cudaStream_t>, HostPipe*>> g_pipes;
HostPipe* pipe_for(cudaStream_t st) {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return nullptr;
  std::lock_guard<std::mutex> g(g_pipes_mu);
  for (auto& kv : g_pipes)
    if (kv.first.first == dev && kv.first.second == st) return kv.second;
  g_pipes.push_back({{dev, st}, new HostPipe()});
  return g_pipes.back().second;
}
// Holds the pipe for one call. Whatever way the call returns, no copy may still be reading or writing the caller's host
// buffers afterwards: the destructor drains the three streams unless the normal path already did.
struct PipeLease {
  HostPipe* pipe;
  cudaStream_t st;
  bool drained = false;
  PipeLease(HostPipe* p, cudaStream_t s) : pipe(p), st(s) { pipe->busy.lock(); }
  ~PipeLease() {
    if (!drained) {
      if (pipe->in) cudaStreamSynchronize(pipe->in);
      cudaStreamSynchronize(st);
      if (pipe->out) cudaStreamSynchronize(pipe->out);
    }
    pipe->busy.unlock();
  }
  cudaError_t drain() {
    cudaError_t e = cudaStreamSynchronize(pipe->out);
    cudaError_t e2 = cudaStreamSynchronize(st);
    drained = true;
    return e != cudaSuccess ? e : e2;
  }
};
int64_t pick_chunks(const fa_problem_t* p, size_t total_bytes) {
  if (p->batch < 2 || total_bytes < (size_t(64) << 20)) return 1;
  return std::min<int64_t>(p->batch, 8);
}
}  // namespace

int fa_forward_host(const fa_problem_t* p, const void* q, const void* k, const void* v, void* o, void* l,
                    void* m, void* dev_arena, size_t dev_arena_bytes, void* stream) {
  Arena a;
  int rc = arena_layout(p, 0, &a);
  if (rc) return rc;
  if (!dev_arena || dev_arena_bytes < a.total) return FA_EINVAL_WORKSPACE;
  if (!q || !k || !v || !o || !l || !m) return FA_EINVAL_NULL;
  if (p->batch == 0) return FA_OK;
  char* base = (char*)dev_arena;
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t B = p->batch;
  const int64_t nch = pick_chunks(p, a.nq_b + a.nk_b + a.nv_b + a.no_b);
  HostPipe* pp = pipe_for(st);
  if (!pp) return FA_ENODEVICE;
  PipeLease lease(pp, st);
  HostPipe& pipe = *pp;
  FA_CU(pipe.reserve(int(2 * nch + 1)));
  FA_CU(cudaEventRecord(pipe.ev[2 * nch], st));          // uploads start after prior work on `stream`
  FA_CU(cudaStreamWaitEvent(pipe.in, pipe.ev[2 * nch], 0));
  const size_t sq = a.nq_b / B, sk = a.nk_b / B, sv = a.nv_b / B, so = a.no_b / B, sl = a.nl_b / B, sm = a.nm_b / B;
  for (int64_t c = 0; c < nch; ++c) {
    const int64_t b0 = B * c / nch, nb = B * (c + 1) / nch - b0;
    FA_CU(cudaMemcpyAsync(base + a.q + b0 * sq, (const char*)q + b0 * sq, nb * sq, cudaMemcpyHostToDevice, pipe.in));
    FA_CU(cudaMemcpyAsync(base + a.k + b0 * sk, (const char*)k + b0 * sk, nb * sk, cudaMemcpyHostToDevice, pipe.in));
    FA_CU(cudaMemcpyAsync(base + a.v + b0 * sv, (const char*)v + b0 * sv, nb * sv, cudaMemcpyHostToDevice, pipe.in));
    if (p->accumulate) {
      FA_CU(cudaMemcpyAsync(base + a.o + b0 * so, (char*)o + b0 * so, nb * so, cudaMemcpyHostToDevice, pipe.in));
      FA_CU(cudaMemcpyAsync(base + a.l + b0 * sl, (char*)l + b0 * sl, nb * sl, cudaMemcpyHostToDevice, pipe.in));
      FA_CU(cudaMemcpyAsync(base + a.m + b0 * sm, (char*)m + b0 * sm, nb * sm, cudaMemcpyHostToDevice, pipe.in));
    }
    FA_CU(cudaEventRecord(pipe.ev[2 * c], pipe.in));
    FA_CU(cudaStreamWaitEvent(st, pipe.ev[2 * c], 0));
    fa_problem_t sub = *p;
    sub.batch = nb;
    rc = fa_forward(&sub, base + a.q + b0 * sq, base + a.k + b0 * sk, base + a.v + b0 * sv, base + a.o + b0 * so,
                    base + a.l + b0 * sl, base + a.m + b0 * sm, base + a.ws, a.total - a.ws, stream);
    if (rc) return rc;
    FA_CU(cudaEventRecord(pipe.ev[2 * c + 1], st));
    FA_CU(cudaStreamWaitEvent(pipe.out, pipe.ev[2 * c + 1], 0));
    FA_CU(cudaMemcpyAsync((char*)o + b0 * so, base + a.o + b0 * so, nb * so, cudaMemcpyDeviceToHost, pipe.out));
    FA_CU(cudaMemcpyAsync((char*)l + b0 * sl, base + a.l + b0 * sl, nb * sl, cudaMemcpyDeviceToHost, pipe.out));
    FA_CU(cudaMemcpyAsync((char*)m + b0 * sm, base + a.m + b0 * sm, nb * sm, cudaMemcpyDeviceToHost, pipe.out));
  }
  FA_CU(lease.drain());
  return FA_OK;
}

}  // extern "C" (the shared body of the two backward host entry points follows)

namespace {
// resident: Q, K, V, O, l, m are already in the arena (left there by fa_forward_host); only dO is uploaded
int backward_host_impl(const fa_problem_t* p, bool resident, const void* q, const void* k, const void* v,
                       const void* o, const void* l, const void* m, const void* d_o, void* d_q, void* d_k, void* d_v,
                       void* dev_arena, size_t dev_arena_bytes, void* stream) {
  Arena a;
  int rc = arena_layout(p, 1, &a);
  if (rc) return rc;
  if (!dev_arena || dev_arena_bytes < a.total) return FA_EINVAL_WORKSPACE;
  if (!resident && (!q || !k || !v || !o || !l || !m)) return FA_EINVAL_NULL;
  if (!d_o || !d_q || !d_k || !d_v) return FA_EINVAL_NULL;
  if (p->batch == 0) return FA_OK;
  char* base = (char*)dev_arena;
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t B = p->batch;
  const int64_t nch = pick_chunks(p, 2 * (a.nq_b + a.nk_b + a.nv_b + a.no_b));
  HostPipe* pp = pipe_for(st);
  if (!pp) return FA_ENODEVICE;
  PipeLease lease(pp, st);
  HostPipe& pipe = *pp;
  FA_CU(pipe.reserve(int(2 * nch + 1)));
  FA_CU(cudaEventRecord(pipe.ev[2 * nch], st));
  FA_CU(cudaStreamWaitEvent(pipe.in, pipe.ev[2 * nch], 0));
  const size_t sq = a.nq_b / B, sk = a.nk_b / B, sv = a.nv_b / B, so = a.no_b / B, sl = a.nl_b / B, sm = a.nm_b / B;
  for (int64_t c = 0; c < nch; ++c) {
    const int64_t b0 = B * c / nch, nb = B * (c + 1) / nch - b0;
    if (!resident) {
      FA_CU(cudaMemcpyAsync(base + a.q + b0 * sq, (const char*)q + b0 * sq, nb * sq, cudaMemcpyHostToDevice, pipe.in));
      FA_CU(cudaMemcpyAsync(base + a.k + b0 * sk, (const char*)k + b0 * sk, nb * sk, cudaMemcpyHostToDevice, pipe.in));
      FA_CU(cudaMemcpyAsync(base + a.v + b0 * sv, (const char*)v + b0 * sv, nb * sv, cudaMemcpyHostToDevice, pipe.in));
      FA_CU(cudaMemcpyAsync(base + a.o + b0 * so, (const char*)o + b0 * so, nb * so, cudaMemcpyHostToDevice, pipe.in));
      FA_CU(cudaMemcpyAsync(base + a.l + b0 * sl, (const char*)l + b0 * sl, nb * sl, cudaMemcpyHostToDevice, pipe.in));
      FA_CU(cudaMemcpyAsync(base + a.m + b0 * sm, (const char*)m + b0 * sm, nb * sm, cudaMemcpyHostToDevice, pipe.in));
    }
    FA_CU(cudaMemcpyAsync(base + a.d_o + b0 * so, (const char*)d_o + b0 * so, nb * so, cudaMemcpyHostToDevice, pipe.in));
    FA_CU(cudaEventRecord(pipe.ev[2 * c], pipe.in));
    FA_CU(cudaStreamWaitEvent(st, pipe.ev[2 * c], 0));
    fa_problem_t sub = *p;
    sub.batch = nb;
    rc = fa_backward(&sub, base + a.q + b0 * sq, base + a.k + b0 * sk, base + a.v + b0 * sv, base + a.o + b0 * so,
                     base + a.l + b0 * sl, base + a.m + b0 * sm, base + a.d_o + b0 * so, base + a.d_q + b0 * sq,
                     base + a.d_k + b0 * sk, base + a.d_v + b0 * sv, base + a.ws, a.total - a.ws, stream);
    if (rc) return rc;
    FA_CU(cudaEventRecord(pipe.ev[2 * c + 1], st));
    FA_CU(cudaStreamWaitEvent(pipe.out, pipe.ev[2 * c + 1], 0));
    FA_CU(cudaMemcpyAsync((char*)d_q + b0 * sq, base + a.d_q + b0 * sq, nb * sq, cudaMemcpyDeviceToHost, pipe.out));
    FA_CU(cudaMemcpyAsync((char*)d_k + b0 * sk, base + a.d_k + b0 * sk, nb * sk, cudaMemcpyDeviceToHost, pipe.out));
    FA_CU(cudaMemcpyAsync((char*)d_v + b0 * sv, base + a.d_v + b0 * sv, nb * sv, cudaMemcpyDeviceToHost, pipe.out));
  }
  FA_CU(lease.drain());
  return FA_OK;
}
}  // namespace

extern "C" {

int fa_backward_host(const fa_problem_t* p, const void* q, const void* k, const void* v, const void* o,
                     const void* l, const void* m, const void* d_o, void* d_q, void* d_k, void* d_v,
                     void* dev_arena, size_t dev_arena_bytes, void* stream) {
  return backward_host_impl(p, false, q, k, v, o, l, m, d_o, d_q, d_k, d_v, dev_arena, dev_arena_bytes, stream);
}

// One training step (forward + gradient) on host buffers, pipelined over batch chunks: upload of chunk c+1 (Q, K, V, dO),
// forward + backward of chunk c and download of chunk c-1 (O, l, m, dQ, dK, dV) overlap, so both PCIe directions are busy
// for the whole step (the two-call sequence is upload-bound in the forward and download-bound in the backward).
size_t fa_step_host_arena_bytes(const fa_problem_t* p) {
  Arena a;
  if (arena_layout(p, 1, &a)) return 0;
  return a.ws + align_up(std::max(fa_workspace_bytes(p, 0), fa_workspace_bytes(p, 1)));
}

int fa_forward_backward_host(const fa_problem_t* p, const void* q, const void* k, const void* v, const void* d_o,
                             void* o, void* l, void* m, void* d_q, void* d_k, void* d_v, void* dev_arena,
                             size_t dev_arena_bytes, void* stream) {
  Arena a;
  int rc = arena_layout(p, 1, &a);
  if (rc) return rc;
  if (p->accumulate) return FA_EINVAL_SHAPE;   // a step starts from fresh outputs
  const size_t need = fa_step_host_arena_bytes(p);
  if (!dev_arena || dev_arena_bytes < need) return FA_EINVAL_WORKSPACE;
  if (!q || !k || !v || !d_o || !o || !l || !m || !d_q || !d_k || !d_v) return FA_EINVAL_NULL;
  if (p->batch == 0) return FA_OK;
  char* base = (char*)dev_arena;
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t B = p->batch;
  // chunks of the batch in flight: fill + drain cost two chunk transfers, so more chunks are better until a chunk's
  // kernels stop filling the GPU (FA_HOST_CHUNKS overrides for A/B runs)
  int64_t want = 16;
  if (const char* e = getenv("FA_HOST_CHUNKS")) want = std::max<int64_t>(1, atoll(e));
  const int64_t nch = p->batch < 2 || a.nq_b + a.nk_b + a.nv_b + a.no_b < (size_t(64) << 20) ? 1 : std::min<int64_t>(B, want);
  HostPipe* pp = pipe_for(st);
  if (!pp) return FA_ENODEVICE;
  PipeLease lease(pp, st);
  HostPipe& pipe = *pp;
  FA_CU(pipe.reserve(int(2 * nch + 1)));
  FA_CU(cudaEventRecord(pipe.ev[2 * nch], st));
  FA_CU(cudaStreamWaitEvent(pipe.in, pipe.ev[2 * nch], 0));
  const size_t sq = a.nq_b / B, sk = a.nk_b / B, sv = a.nv_b / B, so = a.no_b / B, sl = a.nl_b / B, sm = a.nm_b / B;
  for (int64_t c = 0; c < nch; ++c) {
    const int64_t b0 = B * c / nch, nb = B * (c + 1) / nch - b0;
    FA_CU(cudaMemcpyAsync(base + a.q + b0 * sq, (const char*)q + b0 * sq, nb * sq, cudaMemcpyHostToDevice, pipe.in));
    FA_CU(cudaMemcpyAsync(base + a.k + b0 * sk, (const char*)k + b0 * sk, nb * sk, cudaMemcpyHostToDevice, pipe.in));
    FA_CU(cudaMemcpyAsync(base + a.v + b0 * sv, (const char*)v + b0 * sv, nb * sv, cudaMemcpyHostToDevice, pipe.in));
    FA_CU(cudaMemcpyAsync(base + a.d_o + b0 * so, (const char*)d_o + b0 * so, nb * so, cudaMemcpyHostToDevice, pipe.in));
    FA_CU(cudaEventRecord(pipe.ev[2 * c], pipe.in));
    FA_CU(cudaStreamWaitEvent(st, pipe.ev[2 * c], 0));
    fa_problem_t sub = *p;
    sub.batch = nb;
    rc = fa_forward(&sub, base + a.q + b0 * sq, base + a.k + b0 * sk, base + a.v + b0 * sv, base + a.o + b0 * so,
                    base + a.l + b0 * sl, base + a.m + b0 * sm, base + a.ws, need - a.ws, stream);
    if (rc) return rc;
    rc = fa_backward(&sub, base + a.q + b0 * sq, base + a.k + b0 * sk, base + a.v + b0 * sv, base + a.o + b0 * so,
                     base + a.l + b0 * sl, base + a.m + b0 * sm, base + a.d_o + b0 * so, base + a.d_q + b0 * sq,
                     base + a.d_k + b0 * sk, base + a.d_v + b0 * sv, base + a.ws, need - a.ws, stream);
    if (rc) return rc;
    FA_CU(cudaEventRecord(pipe.ev[2 * c + 1], st));
    FA_CU(cudaStreamWaitEvent(pipe.out, pipe.ev[2 * c + 1], 0));
    FA_CU(cudaMemcpyAsync((char*)o + b0 * so, base + a.o + b0 * so, nb * so, cudaMemcpyDeviceToHost, pipe.out));
    FA_CU(cudaMemcpyAsync((char*)l + b0 * sl, base + a.l + b0 * sl, nb * sl, cudaMemcpyDeviceToHost, pipe.out));
    FA_CU(cudaMemcpyAsync((char*)m + b0 * sm, base + a.m + b0 * sm, nb * sm, cudaMemcpyDeviceToHost, pipe.out));
    FA_CU(cudaMemcpyAsync((char*)d_q + b0 * sq, base + a.d_q + b0 * sq, nb * sq, cudaMemcpyDeviceToHost, pipe.out));
    FA_CU(cudaMemcpyAsync((char*)d_k + b0 * sk, base + a.d_k + b0 * sk, nb * sk, cudaMemcpyDeviceToHost, pipe.out));
    FA_CU(cudaMemcpyAsync((char*)d_v + b0 * sv, base + a.d_v + b0 * sv, nb * sv, cudaMemcpyDeviceToHost, pipe.out));
  }
  FA_CU(lease.drain());
  return FA_OK;
}

int fa_backward_host_resident(const fa_problem_t* p, const void* d_o, void* d_q, void* d_k, void* d_v,
                              void* dev_arena, size_t dev_arena_bytes, void* stream) {
  return backward_host_impl(p, true, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, d_o, d_q, d_k, d_v,
                            dev_arena, dev_arena_bytes, stream);
}

}  // extern "C"
