// fa_launch.h — internal contract between the C-ABI front (fa_api.cu) and the kernel
// families. Not installed; the public surface is include/fa_b200.h.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#include <algorithm>

#include "fa_rules.h"

namespace fa {

struct LaunchArgs {
  int32_t dtype;  // 0 f16, 1 f32, 2 f64
  int32_t d, v_d;
  int64_t batch;
  int32_t accumulate;
  FaRule rule;
  const void *q, *k, *v;
  void *o, *l, *m;                // forward outputs / backward inputs
  const void* d_o;
  const void* prep_d_o;  // dense dO for the statistics pass (d_o itself may point at a pitch-padded copy)
  void *d_q, *d_k, *d_v;
  void* workspace;
  size_t workspace_bytes;
  int32_t partial_keys;  // the call covers a shard of the keys only (ring): no per-row renormalisation in the backward
  // elements between consecutive channel rows of the q-length tensors (Q, O, dO, dQ) and the k-length tensors (K, V, dK,
  // dV); 0 = dense (the sequence length). Set by the pitch-padding pack pass (fa_pack.cu) for lengths that are not
  // multiples of 8 halves, which TMA cannot address directly (row pitch must be a multiple of 16 bytes).
  int64_t q_pitch, k_pitch;
  // 0 = channel-first [batch][channels][sequence] (the reference's layout); 1 = channel-last
  // [outer][sequence][heads][channels] with batch = outer * heads (fp16 tcgen05 kernels only; l, m stay [batch][q])
  int32_t layout, heads;
  // fa_backward_accumulate: d_q is an fp32 accumulator that dQ is ADDED into; problem pb adds into accumulator element
  // pb % dq_fold. fp16 fused head_dim-128 backward only.
  int32_t grad_acc;
  int64_t dq_fold;
  int32_t grad_split;  // fp16 backward: dS handed to the tensor cores as hi + lo fp16 pairs (fa_set_grad_precision)
  int32_t variant;  // fa_set_path_override value (0 auto; 4 = fp16 backward as two kernels; 5 / 6 = forward tile configuration)
};

void count_launch();

// Counts one kernel launch and, when kernel timing is on (fa_kernel_timing), brackets it with
// CUDA events on the launching stream so that bench.py can report per-kernel durations.
struct ScopedKernel {
  ScopedKernel(const char* name, cudaStream_t stream);
  ~ScopedKernel();
  cudaStream_t stream_;
  int slot_;
};

// generic SIMT family (fa_generic.cu). Any channel count; above 256 channels the grid (batch x row tiles x channel
// slices) must fit 31 bits, for the forward or for both backward kernels.
bool generic_supports(const LaunchArgs& a, bool backward);
size_t generic_workspace_bytes(int dtype, int64_t batch, int64_t nq, bool backward);
cudaError_t generic_forward(const LaunchArgs& a, cudaStream_t stream);
cudaError_t generic_backward(const LaunchArgs& a, cudaStream_t stream);

// partial-result algebra for K/V-ring sharding (fa_partial.cu)
cudaError_t partial_merge(const LaunchArgs& a, const void* o_part, const void* l_part, const void* m_part,
                          void* o_acc, void* l_acc, void* m_acc, int first, cudaStream_t stream);
cudaError_t partial_finalize(const LaunchArgs& a, const void* o_acc, const void* l_acc, const void* m_acc, void* o,
                             void* l, void* m, cudaStream_t stream);

// gradient shards of the ring backward: acc (float; double for f64) (+)= part, and the final cast
cudaError_t grad_accumulate(int dtype, const void* part, void* acc, int64_t n, int first, cudaStream_t stream);
cudaError_t grad_finalize(int dtype, const void* acc, void* out, int64_t n, cudaStream_t stream);

// channel-last <-> channel-first adapter (fa_layout.cu)
cudaError_t layout_transpose(int dtype, const void* x, void* y, int64_t B, int64_t S, int32_t H, int32_t C,
                             int to_channel_first, int variant, cudaStream_t stream);

// pitch-padding copies for the TMA paths (fa_pack.cu): rows of `len` elements, source / destination pitches in elements
cudaError_t pack_rows(int elt_bytes, const void* src, void* dst, int64_t rows, int64_t len, int64_t src_pitch,
                      int64_t dst_pitch, cudaStream_t stream);

cudaError_t pack_channels_f32(const float* src, float* dst, int64_t batch, int64_t ch, int64_t len, int64_t src_ch,
                              int64_t src_pitch, int64_t dst_ch, int64_t dst_pitch, cudaStream_t stream);

// tcgen05 / TMEM / TMA family for half (fa_fwd_f16_sm100.cu, fa_bwd_f16_sm100.cu)
bool sm100_f16_forward_supports(const LaunchArgs& a);
bool sm100_f16_backward_supports(const LaunchArgs& a);
bool sm100_f16_backward_accumulate_supports(const LaunchArgs& a);
size_t sm100_f16_workspace_bytes(const LaunchArgs& a, bool backward);
cudaError_t sm100_f16_forward(const LaunchArgs& a, cudaStream_t stream);
cudaError_t sm100_f16_backward(const LaunchArgs& a, cudaStream_t stream);

// tcgen05 kind::tf32 forward for float with a 3xTF32 split (fa_fwd_f32_sm100.cu)
bool sm100_f32_forward_supports(const LaunchArgs& a);
size_t sm100_f32_forward_workspace_bytes(const LaunchArgs& a);
cudaError_t sm100_f32_forward(const LaunchArgs& a, cudaStream_t stream);

// fp32 backward on the tensor cores, three bf16 pieces per operand (fa_bwd_f32_sm100.cu)
bool sm100_f32_backward_supports(const LaunchArgs& a);
size_t sm100_f32_backward_workspace_bytes(const LaunchArgs& a);
cudaError_t sm100_f32_backward(const LaunchArgs& a, cudaStream_t stream);

// fp64 on the FP64 tensor cores (mma.sync.m8n8k4.f64), up to 64 channels (fa_f64_dmma.cu)
bool f64_dmma_forward_supports(const LaunchArgs& a);
cudaError_t f64_dmma_forward(const LaunchArgs& a, cudaStream_t stream);
bool f64_dmma_backward_supports(const LaunchArgs& a);
cudaError_t f64_dmma_backward(const LaunchArgs& a, cudaStream_t stream);

}  // namespace fa
