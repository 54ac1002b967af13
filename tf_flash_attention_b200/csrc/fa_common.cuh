// fa_common.cuh — small shared device/host helpers for all kernel families.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <type_traits>

#include "fa_rules.h"

namespace fa {

template <typename T> struct AccOf { using type = float; };
template <> struct AccOf<double> { using type = double; };
// l is float for half (and bf16), T otherwise (reference: flash_attention.h:181-185)
template <typename T> struct LOf { using type = T; };
template <> struct LOf<__half> { using type = float; };
template <> struct LOf<__nv_bfloat16> { using type = float; };

template <typename T> __device__ __forceinline__ T neg_inf();
template <> __device__ __forceinline__ float neg_inf<float>() { return __int_as_float(0xff800000); }
template <> __device__ __forceinline__ double neg_inf<double>() { return __longlong_as_double(0xfff0000000000000ULL); }

template <typename A, typename T> __device__ __forceinline__ A to_acc(T v) { return static_cast<A>(v); }
template <> __device__ __forceinline__ float to_acc<float, __half>(__half v) { return __half2float(v); }
template <> __device__ __forceinline__ float to_acc<float, __nv_bfloat16>(__nv_bfloat16 v) { return __bfloat162float(v); }

template <typename T, typename A> __device__ __forceinline__ T from_acc(A v) { return static_cast<T>(v); }
template <> __device__ __forceinline__ __half from_acc<__half, float>(float v) { return __float2half_rn(v); }
template <> __device__ __forceinline__ __nv_bfloat16 from_acc<__nv_bfloat16, float>(float v) { return __float2bfloat16_rn(v); }

// The reference's "-inf approximation": every byte 0xFA (type_util.h:43-45,
// flash_attention_forward.cc:360-365). Observable in `m` on fully masked rows.
template <typename T> __device__ __forceinline__ T sentinel();
template <> __device__ __forceinline__ __half sentinel<__half>() { return __ushort_as_half((unsigned short)0xFAFA); }
template <> __device__ __forceinline__ __nv_bfloat16 sentinel<__nv_bfloat16>() {
  return __ushort_as_bfloat16((unsigned short)0xFAFA);
}
template <> __device__ __forceinline__ float sentinel<float>() { return __uint_as_float(0xFAFAFAFAu); }
template <> __device__ __forceinline__ double sentinel<double>() { return __longlong_as_double(0xFAFAFAFAFAFAFAFAULL); }

template <typename T> __device__ __forceinline__ bool is_sentinel(T v);
template <> __device__ __forceinline__ bool is_sentinel<__half>(__half v) { return __half_as_ushort(v) == 0xFAFA; }
template <> __device__ __forceinline__ bool is_sentinel<__nv_bfloat16>(__nv_bfloat16 v) {
  return __bfloat16_as_ushort(v) == 0xFAFA;
}
template <> __device__ __forceinline__ bool is_sentinel<float>(float v) { return __float_as_uint(v) == 0xFAFAFAFAu; }
template <> __device__ __forceinline__ bool is_sentinel<double>(double v) {
  return (unsigned long long)__double_as_longlong(v) == 0xFAFAFAFAFAFAFAFAULL;
}

// two adjacent 16-bit elements (the vectorised passes over fp16 / bf16 tensors)
template <typename T>
using Pair = typename std::conditional<std::is_same<T, __half>::value, __half2, __nv_bfloat162>::type;
__device__ __forceinline__ float2 to_float2(__half2 v) { return __half22float2(v); }
__device__ __forceinline__ float2 to_float2(__nv_bfloat162 v) { return __bfloat1622float2(v); }
__device__ __forceinline__ __half low_of(__half2 v) { return __low2half(v); }
__device__ __forceinline__ __nv_bfloat16 low_of(__nv_bfloat162 v) { return __low2bfloat16(v); }
__device__ __forceinline__ __half high_of(__half2 v) { return __high2half(v); }
__device__ __forceinline__ __nv_bfloat16 high_of(__nv_bfloat162 v) { return __high2bfloat16(v); }
__device__ __forceinline__ __half2 pair_of(__half a, __half b) { return __halves2half2(a, b); }
__device__ __forceinline__ __nv_bfloat162 pair_of(__nv_bfloat16 a, __nv_bfloat16 b) { return __halves2bfloat162(a, b); }
template <typename T> __device__ __forceinline__ Pair<T> pair_rn(float a, float b);
template <> __device__ __forceinline__ __half2 pair_rn<__half>(float a, float b) { return __floats2half2_rn(a, b); }
template <> __device__ __forceinline__ __nv_bfloat162 pair_rn<__nv_bfloat16>(float a, float b) {
  return __floats2bfloat162_rn(a, b);
}

__device__ __forceinline__ float acc_exp(float x) { return expf(x); }
__device__ __forceinline__ double acc_exp(double x) { return exp(x); }
__device__ __forceinline__ float acc_log(float x) { return logf(x); }
__device__ __forceinline__ double acc_log(double x) { return log(x); }
__device__ __forceinline__ float acc_max(float a, float b) { return fmaxf(a, b); }
__device__ __forceinline__ double acc_max(double a, double b) { return fmax(a, b); }

}  // namespace fa
