// fa_layout.cu — layout adapter for the step either side of the attention op (SURVEY.md section 8, f3).
// The reference's README example surrounds the op with einsums that produce / consume the channel-first layout
// [batch, head, channel, seq]; most models keep activations channel-last, [batch, seq, head, channel]. This kernel is
// the HBM-bound transpose between the two (tiles of 64 x 64 or 32 x 32 elements through shared memory, both sides
// coalesced). It is an adapter, not a fusion: reading channel-last tiles directly (K-major operands for Q K^T, the mirrored
// descriptors everywhere else) is a round-2 item (DESIGN.md 6b).
#include "fa_common.cuh"
#include "fa_launch.h"

namespace fa {

// to_channel_first: x [B, S, H, C] -> y [B, H, C, S];  otherwise x [B, H, C, S] -> y [B, S, H, C].
// A tile is (32 V) positions x (32 V) channels; every thread reads and writes V contiguous elements (V = 2: 4-byte
// accesses for half, 8-byte for float, so a warp covers a whole 128 / 256-byte row on both sides). The tile is kept
// element-wise in shared memory with an odd pitch: the vector sits in registers only. One CTA walks TILES_PER_CTA
// consecutive tiles along the sequence and issues the global loads of tile t + 1 before it writes tile t out, so loads
// stay in flight during the store phase (with one tile per CTA the kernel sat at 54 % of the HBM bandwidth, stalled on
// the load latency at the head of every CTA: profiles/r1_layout_ncu.md).
constexpr int LAYOUT_TILES_PER_CTA = 8;

template <typename T, int V, bool TO_CF>
__global__ void __launch_bounds__(256, V == 4 ? 2 : 6) layout_transpose_kernel(const T* __restrict__ x, T* __restrict__ y, int64_t S,
                                                                   int32_t H, int32_t C) {
  constexpr int TD = 32 * V;
  constexpr int R = TD / 8;                            // rows per thread on each side
  struct alignas(sizeof(T) * V) Vec { T e[V]; };
  __shared__ T tile[TD][TD + 1];
  const int64_t bh = blockIdx.x;   // b * H + h
  const int64_t b = bh / H;
  const int32_t h = int32_t(bh - b * H);
  const int32_t c0 = blockIdx.z * TD;
  const int tx = threadIdx.x * V, ty = threadIdx.y;   // 32 x 8 threads
  const int64_t s_first = int64_t(blockIdx.y) * (TD * LAYOUT_TILES_PER_CTA);
  const int ntiles = int(((S - s_first < TD * LAYOUT_TILES_PER_CTA ? S - s_first : TD * LAYOUT_TILES_PER_CTA) + TD - 1) / TD);
  const int64_t hc = int64_t(H) * C;
  // element (s, c): channel-last at cl + s * H * C + c, channel-first at cf + c * S + s
  const T* cl = (TO_CF ? x : y) + (b * S * H + h) * int64_t(C);
  const T* cf = (TO_CF ? y : x) + bh * int64_t(C) * S;
  // rows of the source tile run along positions (channel-last source) or channels (channel-first source); thread (tx, ty)
  // owns column tx of rows ty, ty + 8, ...; the destination tile is the transpose. V > 1 is launched only when C and S
  // are multiples of V: a vector never straddles an edge.
  const int64_t in_row = TO_CF ? hc : S, out_row = TO_CF ? S : hc;           // stride between rows
  const int64_t in_tile = TO_CF ? TD * hc : TD, out_tile = TO_CF ? TD : TD * hc;   // stride between tiles (along s)
  const T* src = TO_CF ? cl + (s_first + ty) * hc + (c0 + tx) : cf + (c0 + ty) * S + (s_first + tx);
  T* dst = const_cast<T*>(TO_CF ? cf + (c0 + ty) * S + (s_first + tx) : cl + (s_first + ty) * hc + (c0 + tx));
  const bool c_col_ok = c0 + tx < C;                    // column predicate of the channel-last side

  Vec regs[R];
  auto load_tile = [&](int64_t s0) {
#pragma unroll
    for (int i = 0; i < R; ++i) {
      const int r = ty + 8 * i;
      const bool ok = TO_CF ? (s0 + r < S && c_col_ok) : (c0 + r < C && s0 + tx < S);
      if (ok) regs[i] = *reinterpret_cast<const Vec*>(src + i * 8 * in_row);
    }
    src += in_tile;
  };

  load_tile(s_first);
#pragma unroll 1
  for (int t = 0; t < ntiles; ++t) {
    const int64_t s0 = s_first + int64_t(t) * TD;
#pragma unroll
    for (int i = 0; i < R; ++i) {
#pragma unroll
      for (int j = 0; j < V; ++j) tile[ty + 8 * i][tx + j] = regs[i].e[j];   // out-of-range entries are never read back
    }
    __syncthreads();
    if (t + 1 < ntiles) load_tile(s0 + TD);   // in flight while this tile is written out
#pragma unroll
    for (int i = 0; i < R; ++i) {
      const int r = ty + 8 * i;
      Vec v;
#pragma unroll
      for (int j = 0; j < V; ++j) v.e[j] = tile[tx + j][r];
      const bool ok = TO_CF ? (c0 + r < C && s0 + tx < S) : (s0 + r < S && c_col_ok);
      if (ok) *reinterpret_cast<Vec*>(dst + i * 8 * out_row) = v;
    }
    dst += out_tile;
    __syncthreads();   // the tile is rewritten at the top of the next iteration
  }
}

template <typename T, int V>
static cudaError_t layout_launch(const void* x, void* y, int64_t B, int64_t S, int32_t H, int32_t C, int to_cf,
                                 cudaStream_t stream) {
  constexpr int TD = 32 * V;
  constexpr int64_t SPAN = int64_t(TD) * LAYOUT_TILES_PER_CTA;
  const dim3 grid(unsigned(B * H), unsigned((S + SPAN - 1) / SPAN), unsigned((C + TD - 1) / TD));
  ScopedKernel timed("layout_transpose", stream);
  if (to_cf) layout_transpose_kernel<T, V, true><<<grid, dim3(32, 8), 0, stream>>>((const T*)x, (T*)y, S, H, C);
  else layout_transpose_kernel<T, V, false><<<grid, dim3(32, 8), 0, stream>>>((const T*)x, (T*)y, S, H, C);
  return cudaGetLastError();
}

// ---- fp16 fast path -------------------------------------------------------------------------------------------------
// The element-wise kernel above is bound by instruction issue for 2-byte elements (one LDS and one STS per element, and
// a warp-tile of 2 KB costs > 300 issued instructions against a budget of ~350 at the HBM roofline). This variant moves
// 4 x 4 blocks of halves through registers: a thread loads four rows of 4 halves (LDG.64), transposes the block with
// eight byte-permutes, stores four 8-byte units (dst row k holds 4 consecutive source rows) and the write side reads
// two units and stores 8 halves (STG.128): 22 memory / permute instructions per 16 elements instead of ~56.
// Shared-memory layout: 64 dst rows x 16 units of 8 bytes, unit index XOR-ed with (dst row / 4): both the unit stores
// (lanes vary the dst row) and the unit loads (lanes vary the unit) are conflict-free (checked on the host for every
// warp: tests/test_capi_host.py::test_layout_fast_path_mapping).
// Requires C % 8 == 0, S % 8 == 0 and 16-byte-aligned bases (vectors then never straddle an edge).
template <bool TO_CF>
__global__ void __launch_bounds__(256, 8) layout_transpose_f16_kernel(const __half* __restrict__ x, __half* __restrict__ y,
                                                                       int64_t S, int32_t H, int32_t C) {
  constexpr int TD = 64;
  __shared__ uint2 tile[TD * 16];
  const int64_t bh = blockIdx.x;   // b * H + h
  const int64_t b = bh / H;
  const int32_t h = int32_t(bh - b * H);
  const int32_t c0 = blockIdx.z * TD;
  const int64_t s_first = int64_t(blockIdx.y) * (TD * LAYOUT_TILES_PER_CTA);
  const int64_t s_left = S - s_first;
  const int ntiles = int(((s_left < TD * LAYOUT_TILES_PER_CTA ? s_left : TD * LAYOUT_TILES_PER_CTA) + TD - 1) / TD);
  const int64_t hc = int64_t(H) * C;
  const __half* cl = (TO_CF ? x : y) + (b * S * H + h) * int64_t(C) + s_first * hc + c0;   // tile origin, channel-last
  const __half* cf = (TO_CF ? y : x) + (bh * C + c0) * S + s_first;                        // tile origin, channel-first
  // source tile: 64 rows (positions when TO_CF, channels otherwise) x 64 contiguous columns; destination = transpose
  const int64_t in_row = TO_CF ? hc : S, out_row = TO_CF ? S : hc;
  const int64_t in_tile = TO_CF ? TD * hc : TD, out_tile = TO_CF ? TD : TD * hc;
  const int tid = threadIdx.x;
  const int kq = tid & 15, rq = tid >> 4;                 // load side: columns 4kq.., rows 4rq..
  const int lane = tid & 31, w = tid >> 5;
  const int u = lane & 7, rsel = lane >> 3;               // store side: 8 source rows 8u.. of two dst rows
  const int rho0 = 16 * (w >> 1) + 4 * rsel + 2 * (w & 1);   // dst rows rho0, rho0 + 1 (same kq' = rho0 / 4)
  const int kqp = rho0 >> 2;
  const __half* src = (TO_CF ? cl : cf) + (4 * rq) * in_row + 4 * kq;
  __half* dst = const_cast<__half*>(TO_CF ? cf : cl) + rho0 * out_row + 8 * u;
  // limits of the CTA's strip in tile coordinates: rows / columns of the SOURCE tile still inside the tensor
  const int c_lim = C - c0 < TD ? C - c0 : TD;            // channels left in this 64-channel slab

  uint2 a[4];
  auto load_tile = [&](int t) {
    const int64_t s_rem = s_left - int64_t(t) * TD;       // positions left from this tile's origin
    const int r_lim = TO_CF ? (s_rem < TD ? int(s_rem) : TD) : c_lim;
    const int k_lim = TO_CF ? c_lim : (s_rem < TD ? int(s_rem) : TD);
    if (r_lim == TD && k_lim == TD) {
#pragma unroll
      for (int j = 0; j < 4; ++j) a[j] = *reinterpret_cast<const uint2*>(src + j * in_row);
    } else {
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (4 * rq + j < r_lim && 4 * kq < k_lim) a[j] = *reinterpret_cast<const uint2*>(src + j * in_row);
    }
    src += in_tile;
  };

  load_tile(0);
#pragma unroll 1
  for (int t = 0; t < ntiles; ++t) {
    // 4 x 4 transpose in registers: unit c = halves (a[0][c], a[1][c], a[2][c], a[3][c])
    uint2 o[4];
    o[0] = make_uint2(__byte_perm(a[0].x, a[1].x, 0x5410), __byte_perm(a[2].x, a[3].x, 0x5410));
    o[1] = make_uint2(__byte_perm(a[0].x, a[1].x, 0x7632), __byte_perm(a[2].x, a[3].x, 0x7632));
    o[2] = make_uint2(__byte_perm(a[0].y, a[1].y, 0x5410), __byte_perm(a[2].y, a[3].y, 0x5410));
    o[3] = make_uint2(__byte_perm(a[0].y, a[1].y, 0x7632), __byte_perm(a[2].y, a[3].y, 0x7632));
#pragma unroll
    for (int c = 0; c < 4; ++c) tile[(4 * kq + c) * 16 + (rq ^ kq)] = o[c];   // out-of-range units are never read back
    __syncthreads();
    if (t + 1 < ntiles) load_tile(t + 1);   // in flight while this tile is written out
    const int64_t s_rem = s_left - int64_t(t) * TD;
    const int r_lim = TO_CF ? (s_rem < TD ? int(s_rem) : TD) : c_lim;   // source rows = destination columns
    const int k_lim = TO_CF ? c_lim : (s_rem < TD ? int(s_rem) : TD);   // source columns = destination rows
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const int rho = rho0 + i;
      const uint2 lo = tile[rho * 16 + ((2 * u) ^ kqp)], hi = tile[rho * 16 + ((2 * u + 1) ^ kqp)];
      if (rho < k_lim && 8 * u < r_lim) *reinterpret_cast<uint4*>(dst + i * out_row) = make_uint4(lo.x, lo.y, hi.x, hi.y);
    }
    dst += out_tile;
    __syncthreads();   // the tile is rewritten at the top of the next iteration
  }
}

static cudaError_t layout_launch_f16(const void* x, void* y, int64_t B, int64_t S, int32_t H, int32_t C, int to_cf,
                                     cudaStream_t stream) {
  constexpr int64_t SPAN = 64 * LAYOUT_TILES_PER_CTA;
  const dim3 grid(unsigned(B * H), unsigned((S + SPAN - 1) / SPAN), unsigned((C + 63) / 64));
  ScopedKernel timed("layout_transpose_f16", stream);
  if (to_cf) layout_transpose_f16_kernel<true><<<grid, 256, 0, stream>>>((const __half*)x, (__half*)y, S, H, C);
  else layout_transpose_f16_kernel<false><<<grid, 256, 0, stream>>>((const __half*)x, (__half*)y, S, H, C);
  return cudaGetLastError();
}

template <typename T>
static cudaError_t layout_t(const void* x, void* y, int64_t B, int64_t S, int32_t H, int32_t C, int to_cf, int variant,
                            cudaStream_t stream) {
  if (B * S * H * C == 0) return cudaSuccess;
  // V elements per thread when both layouts keep the vectors aligned (C and S multiples of V, V-element-aligned bases);
  // variant (fa_set_path_override, developer A/B): 7 = element-wise kernel with pairs, 8 = one element per thread,
  // 9 = four halves per thread
  const auto aligned = [&](int v) {
    return C % v == 0 && S % v == 0 &&
           (reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(y)) % (v * sizeof(T)) == 0;
  };
  if constexpr (sizeof(T) == 2) {
    if (variant == 9 && aligned(4)) return layout_launch<T, 4>(x, y, B, S, H, C, to_cf, stream);
    if (variant != 8 && variant != 7 && aligned(8)) return layout_launch_f16(x, y, B, S, H, C, to_cf, stream);
  }
  if constexpr (sizeof(T) < 8) {
    if (variant != 8 && aligned(2)) return layout_launch<T, 2>(x, y, B, S, H, C, to_cf, stream);
  }
  return layout_launch<T, 1>(x, y, B, S, H, C, to_cf, stream);
}

cudaError_t layout_transpose(int dtype, const void* x, void* y, int64_t B, int64_t S, int32_t H, int32_t C,
                             int to_channel_first, int variant, cudaStream_t stream) {
  switch (dtype) {
    case 0:
    case 3:   // bf16 moves the same 2-byte words: the fp16 kernels on reinterpreted pointers, bit-exact
      return layout_t<__half>(x, y, B, S, H, C, to_channel_first, variant, stream);
    case 1: return layout_t<float>(x, y, B, S, H, C, to_channel_first, variant, stream);
    default: return layout_t<double>(x, y, B, S, H, C, to_channel_first, variant, stream);
  }
}

}  // namespace fa
