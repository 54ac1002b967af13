// fa_partial.cu — merging partial attention results over disjoint key shards (K/V ring support).
// New functionality (the reference is single-GPU): when one long sequence is sharded over GPUs, each
// ring step attends the local queries to the visiting K/V shard with fa_forward (global index bases
// in fa_problem_t) and the partial (O, l, m) is folded into fp32 accumulators with the usual online
// softmax algebra; fa_partial_finalize then emits O, l, m in the reference's output contract.
#include "fa_common.cuh"
#include "fa_launch.h"

#include <type_traits>

namespace fa {

template <typename T, typename A>
__global__ void partial_merge_kernel(const T* __restrict__ o_part, const typename LOf<T>::type* __restrict__ l_part,
                                     const T* __restrict__ m_part, A* __restrict__ o_acc, A* __restrict__ l_acc,
                                     A* __restrict__ m_acc, int64_t batch, int32_t v_d, int32_t nq, int first) {
  const int64_t total = batch * nq;
  for (int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; i < total; i += int64_t(gridDim.x) * blockDim.x) {
    const int64_t b = i / nq, r = i - b * nq;
    const T mp_t = m_part[i];
    const A lp = A(l_part[i]);
    const bool part_empty = is_sentinel<T>(mp_t) || !(lp > A(0));
    const A mp = part_empty ? neg_inf<A>() : to_acc<A>(mp_t);
    const A ma = first ? neg_inf<A>() : m_acc[i];
    const A la = first ? A(0) : l_acc[i];
    const A m_new = acc_max(ma, mp);
    A wa = A(0), wp = A(0);
    if (m_new != neg_inf<A>()) {
      wa = ma == neg_inf<A>() ? A(0) : acc_exp(ma - m_new);
      wp = part_empty ? A(0) : acc_exp(mp - m_new) * lp;
    }
    m_acc[i] = m_new;
    l_acc[i] = la * wa + wp;
    const T* op = o_part + b * v_d * int64_t(nq) + r;
    A* oa = o_acc + b * v_d * int64_t(nq) + r;
    for (int c = 0; c < v_d; ++c) {
      const A prev = first ? A(0) : oa[int64_t(c) * nq];
      oa[int64_t(c) * nq] = prev * wa + to_acc<A>(op[int64_t(c) * nq]) * wp;
    }
  }
}

template <typename T, typename A>
__global__ void partial_finalize_kernel(const A* __restrict__ o_acc, const A* __restrict__ l_acc,
                                        const A* __restrict__ m_acc, T* __restrict__ o,
                                        typename LOf<T>::type* __restrict__ l, T* __restrict__ m, int64_t batch,
                                        int32_t v_d, int32_t nq) {
  using L = typename LOf<T>::type;
  const int64_t total = batch * nq;
  for (int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; i < total; i += int64_t(gridDim.x) * blockDim.x) {
    const int64_t b = i / nq, r = i - b * nq;
    const A la = l_acc[i], ma = m_acc[i];
    const bool empty = !(la > A(0));
    const A inv = empty ? A(0) : A(1) / la;
    if (empty) {
      m[i] = sentinel<T>();
      l[i] = L(0);
    } else {
      const T m_t = from_acc<T>(ma);
      m[i] = m_t;
      l[i] = L(la * acc_exp(ma - to_acc<A>(m_t)));
    }
    const A* oa = o_acc + b * v_d * int64_t(nq) + r;
    T* og = o + b * v_d * int64_t(nq) + r;
    for (int c = 0; c < v_d; ++c) og[int64_t(c) * nq] = from_acc<T>(oa[int64_t(c) * nq] * inv);
  }
}

// fp16 / bf16 ring traffic (the C5 configuration): two adjacent query rows per thread, so that every access is a 4-byte
// (half2 / bfloat162) or 8-byte (float2) word per lane - twice the bytes in flight of the scalar kernels above, which
// these passes (pure HBM streaming) need. Rows are paired inside one batch element (nq even).
template <typename T>
__global__ void partial_merge_h2_kernel(const Pair<T>* __restrict__ o_part, const float2* __restrict__ l_part,
                                        const Pair<T>* __restrict__ m_part, float2* __restrict__ o_acc,
                                        float2* __restrict__ l_acc, float2* __restrict__ m_acc, int64_t batch,
                                        int32_t v_d, int32_t nq2, int first) {
  const int64_t total = batch * nq2;
  for (int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; i < total; i += int64_t(gridDim.x) * blockDim.x) {
    const int64_t b = i / nq2, r = i - b * nq2;
    const Pair<T> mp_h = m_part[i];
    const float2 lp = l_part[i];
    const float2 ma = first ? make_float2(neg_inf<float>(), neg_inf<float>()) : m_acc[i];
    const float2 la = first ? make_float2(0.f, 0.f) : l_acc[i];
    float wa[2], wp[2], mn[2], ln[2];
    const T mph[2] = {low_of(mp_h), high_of(mp_h)};
    const float lpv[2] = {lp.x, lp.y}, mav[2] = {ma.x, ma.y}, lav[2] = {la.x, la.y};
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      const bool part_empty = is_sentinel<T>(mph[e]) || !(lpv[e] > 0.f);
      const float mp = part_empty ? neg_inf<float>() : to_acc<float>(mph[e]);
      mn[e] = acc_max(mav[e], mp);
      wa[e] = wp[e] = 0.f;
      if (mn[e] != neg_inf<float>()) {
        wa[e] = mav[e] == neg_inf<float>() ? 0.f : acc_exp(mav[e] - mn[e]);
        wp[e] = part_empty ? 0.f : acc_exp(mp - mn[e]) * lpv[e];
      }
      ln[e] = lav[e] * wa[e] + wp[e];
    }
    m_acc[i] = make_float2(mn[0], mn[1]);
    l_acc[i] = make_float2(ln[0], ln[1]);
    const Pair<T>* op = o_part + b * v_d * int64_t(nq2) + r;
    float2* oa = o_acc + b * v_d * int64_t(nq2) + r;
#pragma unroll 8
    for (int c = 0; c < v_d; ++c) {
      const float2 x = to_float2(op[int64_t(c) * nq2]);
      const float2 prev = first ? make_float2(0.f, 0.f) : oa[int64_t(c) * nq2];
      oa[int64_t(c) * nq2] = make_float2(prev.x * wa[0] + x.x * wp[0], prev.y * wa[1] + x.y * wp[1]);
    }
  }
}

template <typename T>
__global__ void partial_finalize_h2_kernel(const float2* __restrict__ o_acc, const float2* __restrict__ l_acc,
                                           const float2* __restrict__ m_acc, Pair<T>* __restrict__ o,
                                           float2* __restrict__ l, Pair<T>* __restrict__ m, int64_t batch, int32_t v_d,
                                           int32_t nq2) {
  const int64_t total = batch * nq2;
  for (int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; i < total; i += int64_t(gridDim.x) * blockDim.x) {
    const int64_t b = i / nq2, r = i - b * nq2;
    const float2 la = l_acc[i], ma = m_acc[i];
    const float lav[2] = {la.x, la.y}, mav[2] = {ma.x, ma.y};
    float inv[2], lo[2];
    T mo[2];
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      const bool empty = !(lav[e] > 0.f);
      inv[e] = empty ? 0.f : 1.f / lav[e];
      mo[e] = empty ? sentinel<T>() : from_acc<T>(mav[e]);
      lo[e] = empty ? 0.f : lav[e] * acc_exp(mav[e] - to_acc<float>(mo[e]));
    }
    m[i] = pair_of(mo[0], mo[1]);
    l[i] = make_float2(lo[0], lo[1]);
    const float2* oa = o_acc + b * v_d * int64_t(nq2) + r;
    Pair<T>* og = o + b * v_d * int64_t(nq2) + r;
#pragma unroll 8
    for (int c = 0; c < v_d; ++c) {
      const float2 x = oa[int64_t(c) * nq2];
      og[int64_t(c) * nq2] = pair_rn<T>(x.x * inv[0], x.y * inv[1]);
    }
  }
}

static bool al(const void* p, uintptr_t n) { return (reinterpret_cast<uintptr_t>(p) & (n - 1)) == 0; }

template <typename T>
static cudaError_t merge_t(const LaunchArgs& a, const void* o_part, const void* l_part, const void* m_part,
                           void* o_acc, void* l_acc, void* m_acc, int first, cudaStream_t stream) {
  using A = typename AccOf<T>::type;
  const int64_t total = a.batch * a.rule.q.total;
  const int blocks = int(std::min<int64_t>((total + 255) / 256, 148 * 16));
  ScopedKernel timed("partial_merge", stream);
  if constexpr (sizeof(T) == 2) {
    if (a.rule.q.total % 2 == 0 && al(o_part, 4) && al(m_part, 4) && al(l_part, 8) && al(o_acc, 8) && al(l_acc, 8) &&
        al(m_acc, 8)) {
      const int b2 = int(std::min<int64_t>((total / 2 + 255) / 256, 148 * 16));
      partial_merge_h2_kernel<T><<<b2, 256, 0, stream>>>((const Pair<T>*)o_part, (const float2*)l_part,
                                                      (const Pair<T>*)m_part, (float2*)o_acc, (float2*)l_acc,
                                                      (float2*)m_acc, a.batch, a.v_d, a.rule.q.total / 2, first);
      return cudaGetLastError();
    }
  }
  partial_merge_kernel<T, A><<<blocks, 256, 0, stream>>>((const T*)o_part, (const typename LOf<T>::type*)l_part,
                                                         (const T*)m_part, (A*)o_acc, (A*)l_acc, (A*)m_acc, a.batch,
                                                         a.v_d, a.rule.q.total, first);
  return cudaGetLastError();
}

template <typename T>
static cudaError_t finalize_t(const LaunchArgs& a, const void* o_acc, const void* l_acc, const void* m_acc, void* o,
                              void* l, void* m, cudaStream_t stream) {
  using A = typename AccOf<T>::type;
  const int64_t total = a.batch * a.rule.q.total;
  const int blocks = int(std::min<int64_t>((total + 255) / 256, 148 * 16));
  ScopedKernel timed("partial_finalize", stream);
  if constexpr (sizeof(T) == 2) {
    if (a.rule.q.total % 2 == 0 && al(o, 4) && al(m, 4) && al(l, 8) && al(o_acc, 8) && al(l_acc, 8) && al(m_acc, 8)) {
      const int b2 = int(std::min<int64_t>((total / 2 + 255) / 256, 148 * 16));
      partial_finalize_h2_kernel<T><<<b2, 256, 0, stream>>>((const float2*)o_acc, (const float2*)l_acc,
                                                         (const float2*)m_acc, (Pair<T>*)o, (float2*)l, (Pair<T>*)m,
                                                         a.batch, a.v_d, a.rule.q.total / 2);
      return cudaGetLastError();
    }
  }
  partial_finalize_kernel<T, A><<<blocks, 256, 0, stream>>>((const A*)o_acc, (const A*)l_acc, (const A*)m_acc, (T*)o,
                                                            (typename LOf<T>::type*)l, (T*)m, a.batch, a.v_d,
                                                            a.rule.q.total);
  return cudaGetLastError();
}

cudaError_t partial_merge(const LaunchArgs& a, const void* o_part, const void* l_part, const void* m_part,
                          void* o_acc, void* l_acc, void* m_acc, int first, cudaStream_t stream) {
  switch (a.dtype) {
    case 0: return merge_t<__half>(a, o_part, l_part, m_part, o_acc, l_acc, m_acc, first, stream);
    case 3: return merge_t<__nv_bfloat16>(a, o_part, l_part, m_part, o_acc, l_acc, m_acc, first, stream);
    case 1: return merge_t<float>(a, o_part, l_part, m_part, o_acc, l_acc, m_acc, first, stream);
    default: return merge_t<double>(a, o_part, l_part, m_part, o_acc, l_acc, m_acc, first, stream);
  }
}

cudaError_t partial_finalize(const LaunchArgs& a, const void* o_acc, const void* l_acc, const void* m_acc, void* o,
                             void* l, void* m, cudaStream_t stream) {
  switch (a.dtype) {
    case 0: return finalize_t<__half>(a, o_acc, l_acc, m_acc, o, l, m, stream);
    case 3: return finalize_t<__nv_bfloat16>(a, o_acc, l_acc, m_acc, o, l, m, stream);
    case 1: return finalize_t<float>(a, o_acc, l_acc, m_acc, o, l, m, stream);
    default: return finalize_t<double>(a, o_acc, l_acc, m_acc, o, l, m, stream);
  }
}

// ---- gradient shards (ring backward): acc (+)= part, and the final cast ----------------------
template <typename T, typename A>
__global__ void grad_accumulate_kernel(const T* __restrict__ part, A* __restrict__ acc, int64_t n, int first) {
  for (int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; i < n; i += int64_t(gridDim.x) * blockDim.x)
    acc[i] = (first ? A(0) : acc[i]) + to_acc<A>(part[i]);
}
template <typename T, typename A>
__global__ void grad_finalize_kernel(const A* __restrict__ acc, T* __restrict__ out, int64_t n) {
  for (int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; i < n; i += int64_t(gridDim.x) * blockDim.x)
    out[i] = from_acc<T>(acc[i]);
}

// 8 elements per thread: one 16-byte load of 16-bit values, two 16-byte read-modify-writes of floats
template <typename T>
__global__ void grad_accumulate_h8_kernel(const uint4* __restrict__ part, float4* __restrict__ acc, int64_t n8,
                                          int first) {
  for (int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; i < n8; i += int64_t(gridDim.x) * blockDim.x) {
    const uint4 p = part[i];
    const Pair<T>* h = reinterpret_cast<const Pair<T>*>(&p);
    float4 a0 = first ? make_float4(0.f, 0.f, 0.f, 0.f) : acc[2 * i];
    float4 a1 = first ? make_float4(0.f, 0.f, 0.f, 0.f) : acc[2 * i + 1];
    const float2 x0 = to_float2(h[0]), x1 = to_float2(h[1]), x2 = to_float2(h[2]), x3 = to_float2(h[3]);
    a0.x += x0.x; a0.y += x0.y; a0.z += x1.x; a0.w += x1.y;
    a1.x += x2.x; a1.y += x2.y; a1.z += x3.x; a1.w += x3.y;
    acc[2 * i] = a0;
    acc[2 * i + 1] = a1;
  }
}
template <typename T>
__global__ void grad_finalize_h8_kernel(const float4* __restrict__ acc, uint4* __restrict__ out, int64_t n8) {
  for (int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; i < n8; i += int64_t(gridDim.x) * blockDim.x) {
    const float4 a0 = acc[2 * i], a1 = acc[2 * i + 1];
    uint4 o;
    Pair<T>* h = reinterpret_cast<Pair<T>*>(&o);
    h[0] = pair_rn<T>(a0.x, a0.y);
    h[1] = pair_rn<T>(a0.z, a0.w);
    h[2] = pair_rn<T>(a1.x, a1.y);
    h[3] = pair_rn<T>(a1.z, a1.w);
    out[i] = o;
  }
}

template <typename T, typename A>
static cudaError_t grad_acc_t(const void* part, void* acc, int64_t n, int first, cudaStream_t stream) {
  if (n == 0) return cudaSuccess;
  const int blocks = int(std::min<int64_t>((n + 255) / 256, 148 * 16));
  ScopedKernel timed("grad_accumulate", stream);
  if constexpr (sizeof(T) == 2) {
    if (n % 8 == 0 && al(part, 16) && al(acc, 16)) {
      const int b8 = int(std::min<int64_t>((n / 8 + 255) / 256, 148 * 16));
      grad_accumulate_h8_kernel<T><<<b8, 256, 0, stream>>>((const uint4*)part, (float4*)acc, n / 8, first);
      return cudaGetLastError();
    }
  }
  grad_accumulate_kernel<T, A><<<blocks, 256, 0, stream>>>((const T*)part, (A*)acc, n, first);
  return cudaGetLastError();
}
template <typename T, typename A>
static cudaError_t grad_fin_t(const void* acc, void* out, int64_t n, cudaStream_t stream) {
  if (n == 0) return cudaSuccess;
  const int blocks = int(std::min<int64_t>((n + 255) / 256, 148 * 16));
  ScopedKernel timed("grad_finalize", stream);
  if constexpr (sizeof(T) == 2) {
    if (n % 8 == 0 && al(acc, 16) && al(out, 16)) {
      const int b8 = int(std::min<int64_t>((n / 8 + 255) / 256, 148 * 16));
      grad_finalize_h8_kernel<T><<<b8, 256, 0, stream>>>((const float4*)acc, (uint4*)out, n / 8);
      return cudaGetLastError();
    }
  }
  grad_finalize_kernel<T, A><<<blocks, 256, 0, stream>>>((const A*)acc, (T*)out, n);
  return cudaGetLastError();
}

cudaError_t grad_accumulate(int dtype, const void* part, void* acc, int64_t n, int first, cudaStream_t stream) {
  switch (dtype) {
    case 0: return grad_acc_t<__half, float>(part, acc, n, first, stream);
    case 3: return grad_acc_t<__nv_bfloat16, float>(part, acc, n, first, stream);
    case 1: return grad_acc_t<float, float>(part, acc, n, first, stream);
    default: return grad_acc_t<double, double>(part, acc, n, first, stream);
  }
}
cudaError_t grad_finalize(int dtype, const void* acc, void* out, int64_t n, cudaStream_t stream) {
  switch (dtype) {
    case 0: return grad_fin_t<__half, float>(acc, out, n, stream);
    case 3: return grad_fin_t<__nv_bfloat16, float>(acc, out, n, stream);
    case 1: return grad_fin_t<float, float>(acc, out, n, stream);
    default: return grad_fin_t<double, double>(acc, out, n, stream);
  }
}

}  // namespace fa
