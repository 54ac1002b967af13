// fa_generic.cu — the any-shape / any-dtype kernel family (SIMT, fp32 or fp64 accumulate).
//
// This is the engine's universal path: it accepts every (q, k, d, v_d) the reference
// accepts, every rule and sync mode, half/float/double, and is what the tcgen05 kernels
// fall back to for shapes TMA cannot address. Up to 256 channels a CTA keeps whole
// [channels][tile] operand tiles in shared memory. Above 256 channels (KC > 0, "wide") the
// same kernels stream the Q.K^T and dO.V^T reductions through shared memory in chunks of
// KC channels and split the output channels across the grid: each CTA owns a slice of at
// most 256 of them and recomputes S for it. Every output element has one writer.
// It is a flash-attention-2 style design (one CTA per Q tile, online softmax in registers, O written once) instead of
// the reference's K-outer loop with O/l/m read-modify-written in HBM under a spin lock
// (reference: flash_attention/kernel/flash_attention.cu:858-1076, 1725-1950).
//
// Semantics preserved from the reference:
//   scale 1/sqrt(d)                      flash_attention.cu:2162
//   padding rule q<size && k<size        flash_attention.cu:927
//   P = exp(s*scale - m) / l             flash_attention.cu:1838-1841
//   dS = P * (dP - D) * scale            flash_attention.cu:1544-1546
//   fully masked rows: O=0, l=0, m=0xFA… flash_attention_forward.cc:352-365
#include "fa_common.cuh"
#include "fa_launch.h"
#include "fa_plan.h"

namespace fa {
namespace generic {

constexpr int NT = 256;  // 16 x 16 thread grid

template <typename T>
struct FwdParams {
  const T* q; const T* k; const T* v;
  T* o; typename LOf<T>::type* l; T* m;
  int32_t d, v_d, nq, nk, n_rtiles;
  int64_t batch;
  int32_t accumulate;
  FaRule rule;
  // wide kernels (KC > 0): the grid runs slices slice_lo .. slice_lo + n_sl - 1 of O's channels, sw channels each;
  // res = Q stays resident in shared memory whole instead of streamed in chunks
  int32_t sw, n_sl, slice_lo, res;
};

template <typename T>
struct BwdParams {
  const T* q; const T* k; const T* v; const T* d_o;
  T* d_q; T* d_k; T* d_v;
  const typename AccOf<T>::type* lse;   // [batch, nq]  m + log(l)  (+inf on empty rows)
  const typename AccOf<T>::type* dsum;  // [batch, nq]  rowsum(dO * O)
  int32_t d, v_d, nq, nk, n_rtiles;
  int64_t batch;
  FaRule rule;
  // wide kernels (KC > 0). dQ: n_sl slices of d, sw channels each. dK/dV: slices 0 .. n_sl_k - 1 cover dK (sw channels
  // each), the remaining n_sl - n_sl_k cover dV (sw_v channels each). res = the resident-side operands (Q and dO, or K
  // and V) stay in shared memory whole instead of streamed in chunks
  int32_t sw, sw_v, n_sl, n_sl_k, res;
};

// ---- tile primitives ---------------------------------------------------------------------
// Thread (ty, tx) of the 16x16 grid owns resident rows ty*RM..ty*RM+RM-1 (contiguous) and
// streamed columns tx + 16*j (interleaved -> conflict-free reads of the +1 padded tile).

// ADD = true adds to acc instead of overwriting it (one channel chunk of a longer reduction).
template <typename A, int BM, int BN, bool ADD = false>
__device__ __forceinline__ void gemm_s(const A* __restrict__ R, const A* __restrict__ S, int C,
                                       A (&acc)[BM / 16][BN / 16], int ty, int tx) {
  constexpr int RM = BM / 16, CN = BN / 16;
  if constexpr (!ADD) {
#pragma unroll
    for (int i = 0; i < RM; ++i)
#pragma unroll
      for (int j = 0; j < CN; ++j) acc[i][j] = A(0);
  }
  for (int c = 0; c < C; ++c) {
    A a[RM], b[CN];
#pragma unroll
    for (int i = 0; i < RM; ++i) a[i] = R[c * BM + ty * RM + i];
#pragma unroll
    for (int j = 0; j < CN; ++j) b[j] = S[c * (BN + 1) + tx + 16 * j];
#pragma unroll
    for (int i = 0; i < RM; ++i)
#pragma unroll
      for (int j = 0; j < CN; ++j) acc[i][j] += a[i] * b[j];
  }
}

// out[i][s] += sum_kk P[row_i][kk] * B[tx+16s][kk]   (B is [NC][BN+1])
template <typename A, int BM, int BN, int NS>
__device__ __forceinline__ void gemm_pv(const A* __restrict__ P, const A* __restrict__ B, int NC,
                                        A (&out)[BM / 16][NS], int ty, int tx) {
  constexpr int RM = BM / 16;
  const A* brow[NS];
  bool bval[NS];
#pragma unroll
  for (int s = 0; s < NS; ++s) {
    int ch = tx + 16 * s;
    bval[s] = ch < NC;
    brow[s] = B + (bval[s] ? ch : 0) * (BN + 1);
  }
  for (int kk = 0; kk < BN; ++kk) {
    A pv[RM];
#pragma unroll
    for (int i = 0; i < RM; ++i) pv[i] = P[(ty * RM + i) * (BN + 1) + kk];
#pragma unroll
    for (int s = 0; s < NS; ++s) {
      A b = bval[s] ? brow[s][kk] : A(0);
#pragma unroll
      for (int i = 0; i < RM; ++i) out[i][s] += pv[i] * b;
    }
  }
}

// loads a [C][W] tile of a channel-first tensor (row pitch n) starting at column x0 into
// smem with row pitch `pitch`, zero-filling columns >= n. Coalesced along the sequence.
template <typename T, typename A>
__device__ __forceinline__ void load_tile(A* __restrict__ dst, const T* __restrict__ src, int C, int W,
                                          int pitch, int64_t n, int64_t x0) {
  const int total = C * W;
  for (int idx = threadIdx.x; idx < total; idx += NT) {
    int c = idx / W, x = idx - c * W;
    int64_t gx = x0 + x;
    dst[c * pitch + x] = gx < n ? to_acc<A>(src[int64_t(c) * n + gx]) : A(0);
  }
}

// acc = R . S^T over C channels in chunks of KC (wide kernels). R is the resident side ([C][BM] already in Rs when
// r_res, else streamed through Rs as [KC][BM] chunks from r_src, row pitch r_n, columns r0..); S is streamed through
// Ss as [KC][BN+1] chunks. Synchronises before each chunk, so the caller need not free Rs / Ss first. Every CTA that
// computes the same tile runs the same products in the same order, so the result is bit-identical across slices.
template <typename T, typename A, int BM, int BN, int KC>
__device__ __forceinline__ void gemm_s_chunked(A* __restrict__ Rs, bool r_res, const T* __restrict__ r_src,
                                               int64_t r_n, int64_t r0, A* __restrict__ Ss,
                                               const T* __restrict__ s_src, int64_t s_n, int64_t s0, int C,
                                               A (&acc)[BM / 16][BN / 16], int ty, int tx) {
#pragma unroll
  for (int i = 0; i < BM / 16; ++i)
#pragma unroll
    for (int j = 0; j < BN / 16; ++j) acc[i][j] = A(0);
  for (int c0 = 0; c0 < C; c0 += KC) {
    const int cc = min(KC, C - c0);
    __syncthreads();
    if (!r_res) load_tile<T, A>(Rs, r_src + int64_t(c0) * r_n, cc, BM, BM, r_n, r0);
    load_tile<T, A>(Ss, s_src + int64_t(c0) * s_n, cc, BN, BN + 1, s_n, s0);
    __syncthreads();
    gemm_s<A, BM, BN, true>(r_res ? Rs + c0 * BM : Rs, Ss, cc, acc, ty, tx);
  }
}

template <typename A>
__device__ __forceinline__ A half_warp_max(A v) {
#pragma unroll
  for (int o = 1; o < 16; o <<= 1) v = acc_max(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
template <typename A>
__device__ __forceinline__ A half_warp_sum(A v) {
#pragma unroll
  for (int o = 1; o < 16; o <<= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// ---- forward -----------------------------------------------------------------------------
// KC == 0: one CTA per Q tile, all v_d output channels. KC > 0 (wide): one CTA per (Q tile, slice of O's channels).
template <typename T, int BM, int BN, int NS, int KC = 0>
__global__ void __launch_bounds__(NT) fwd_kernel(const FwdParams<T> p) {
  using A = typename AccOf<T>::type;
  using L = typename LOf<T>::type;
  constexpr int RM = BM / 16, CN = BN / 16;
  constexpr bool WIDE = KC > 0;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  A* Qs = reinterpret_cast<A*>(smem_raw);                     // [d][BM]     (wide, streamed: [KC][BM])
  A* Ks = Qs + (WIDE && !p.res ? KC : p.d) * BM;              // [d][BN+1]   (wide: [KC][BN+1] chunks)
  A* Vs = Ks + (WIDE ? KC : p.d) * (BN + 1);                  // [v_d][BN+1] (wide: [sw][BN+1])  also the O staging buffer
  A* Ps = Vs + (WIDE ? p.sw : p.v_d) * (BN + 1);              // [BM][BN+1]

  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int rt = p.n_rtiles - 1 - int(blockIdx.x % p.n_rtiles);  // heavy (late) tiles first
  int64_t b = blockIdx.x / p.n_rtiles;
  int slice = 0, c_lo = 0, c_n = 0;  // wide: this CTA's output channels are c_lo .. c_lo + c_n - 1
  if constexpr (WIDE) {
    slice = p.slice_lo + int(b % p.n_sl);
    b /= p.n_sl;
    c_lo = slice * p.sw;
    c_n = min(p.sw, p.v_d - c_lo);
  }
  const int q0 = rt * BM;
  const int q_hi = min(q0 + BM, p.nq) - 1;
  const FaRule& rule = p.rule;
  const A scale = A(1) / sqrt(A(p.d));

  if (!WIDE || p.res) load_tile<T, A>(Qs, p.q + b * p.d * int64_t(p.nq), p.d, BM, BM, p.nq, q0);

  FaPos qpos[RM];
  A m_i[RM], l_i[RM], acc[RM][NS];
#pragma unroll
  for (int i = 0; i < RM; ++i) {
    int qi = min(q0 + ty * RM + i, p.nq - 1);
    qpos[i] = fa_pos(rule, rule.q, qi);
    m_i[i] = neg_inf<A>();
    l_i[i] = A(0);
#pragma unroll
    for (int s = 0; s < NS; ++s) acc[i][s] = A(0);
  }
  if (p.accumulate) {
#pragma unroll
    for (int i = 0; i < RM; ++i) {
      int qi = q0 + ty * RM + i;
      if (qi < p.nq) {
        T mv = p.m[b * p.nq + qi];
        if (!is_sentinel<T>(mv)) {
          m_i[i] = to_acc<A>(mv);
          l_i[i] = A(p.l[b * p.nq + qi]);
#pragma unroll
          for (int s = 0; s < NS; ++s) {
            int ch = tx + 16 * s;
            if (ch < (WIDE ? c_n : p.v_d))
              acc[i][s] = to_acc<A>(p.o[(b * p.v_d + (WIDE ? c_lo + ch : ch)) * int64_t(p.nq) + qi]) * l_i[i];
          }
        }
      }
    }
  }

  int kt_first, kt_last;
  fa_k_tile_range(rule, q0, q_hi, BN, &kt_first, &kt_last);
  for (int kt = kt_first; kt <= kt_last; ++kt) {
    const int k0 = kt * BN;
    const int k_hi = min(k0 + BN, p.nk) - 1;
    const int cls = fa_classify(rule, q0, q_hi, k0, k_hi);
    if (cls == FA_TILE_SKIP) continue;
    __syncthreads();
    A s[RM][CN];
    if constexpr (!WIDE) {
      load_tile<T, A>(Ks, p.k + b * p.d * int64_t(p.nk), p.d, BN, BN + 1, p.nk, k0);
      load_tile<T, A>(Vs, p.v + b * p.v_d * int64_t(p.nk), p.v_d, BN, BN + 1, p.nk, k0);
      __syncthreads();
      gemm_s<A, BM, BN>(Qs, Ks, p.d, s, ty, tx);
    } else {
      load_tile<T, A>(Vs, p.v + (b * p.v_d + c_lo) * int64_t(p.nk), c_n, BN, BN + 1, p.nk, k0);
      gemm_s_chunked<T, A, BM, BN, KC>(Qs, p.res, p.q + b * p.d * int64_t(p.nq), p.nq, q0, Ks,
                                       p.k + b * p.d * int64_t(p.nk), p.nk, k0, p.d, s, ty, tx);
    }

#pragma unroll
    for (int j = 0; j < CN; ++j) {
      const int kj = k0 + tx + 16 * j;
      const bool kvalid = kj < p.nk;
      const FaPos kpos = fa_pos(rule, rule.k, kvalid ? kj : p.nk - 1);
#pragma unroll
      for (int i = 0; i < RM; ++i) {
        bool ok = kvalid && (cls == FA_TILE_FULL || fa_attend(rule, qpos[i], kpos));
        s[i][j] = ok ? s[i][j] * scale : neg_inf<A>();
      }
    }
#pragma unroll
    for (int i = 0; i < RM; ++i) {
      A mx = s[i][0];
#pragma unroll
      for (int j = 1; j < CN; ++j) mx = acc_max(mx, s[i][j]);
      mx = half_warp_max(mx);
      const A m_new = acc_max(m_i[i], mx);
      A alpha = A(1), sum = A(0);
      if (m_new == neg_inf<A>()) {
#pragma unroll
        for (int j = 0; j < CN; ++j) s[i][j] = A(0);
      } else {
        alpha = acc_exp(m_i[i] - m_new);  // exp(-inf) = 0 on the first live tile
#pragma unroll
        for (int j = 0; j < CN; ++j) {
          s[i][j] = acc_exp(s[i][j] - m_new);
          sum += s[i][j];
        }
      }
      sum = half_warp_sum(sum);
      l_i[i] = l_i[i] * alpha + sum;
      m_i[i] = m_new;
#pragma unroll
      for (int sidx = 0; sidx < NS; ++sidx) acc[i][sidx] *= alpha;
#pragma unroll
      for (int j = 0; j < CN; ++j) Ps[(ty * RM + i) * (BN + 1) + tx + 16 * j] = s[i][j];
    }
    __syncthreads();
    gemm_pv<A, BM, BN, NS>(Ps, Vs, WIDE ? c_n : p.v_d, acc, ty, tx);
  }

  // epilogue: O = acc / l staged through smem so that the store is coalesced along q
  __syncthreads();
  A* Os = Vs;  // [c_n][BM+1]  (BM == BN)
#pragma unroll
  for (int i = 0; i < RM; ++i) {
    const A inv = l_i[i] > A(0) ? A(1) / l_i[i] : A(0);
#pragma unroll
    for (int s = 0; s < NS; ++s) {
      int ch = tx + 16 * s;
      if (ch < (WIDE ? c_n : p.v_d)) Os[ch * (BM + 1) + ty * RM + i] = acc[i][s] * inv;
    }
    const int qi = q0 + ty * RM + i;
    // every slice computes the same m and l bit for bit; slice 0 stores them
    if (tx == 0 && qi < p.nq && (!WIDE || slice == 0)) {
      if (l_i[i] > A(0)) {
        // m is stored in T; l is re-expressed against the rounded m so that
        // exp(s - m_T) / l_out reproduces the exact probabilities in the backward.
        const T m_t = from_acc<T>(m_i[i]);
        const A m_back = to_acc<A>(m_t);
        p.m[b * p.nq + qi] = m_t;
        p.l[b * p.nq + qi] = L(l_i[i] * acc_exp(m_i[i] - m_back));
      } else {
        p.m[b * p.nq + qi] = sentinel<T>();
        p.l[b * p.nq + qi] = L(0);
      }
    }
  }
  __syncthreads();
  T* og = p.o + (WIDE ? b * p.v_d + c_lo : b * p.v_d) * int64_t(p.nq);
  const int total = (WIDE ? c_n : p.v_d) * BM;
  for (int idx = threadIdx.x; idx < total; idx += NT) {
    int ch = idx / BM, r = idx - ch * BM;
    if (q0 + r < p.nq) og[int64_t(ch) * p.nq + q0 + r] = from_acc<T>(Os[ch * (BM + 1) + r]);
  }
}

// ---- backward preprocess: LSE and D ------------------------------------------------------
template <typename T>
__global__ void bwd_prep_kernel(const T* __restrict__ o, const T* __restrict__ d_o,
                                const typename LOf<T>::type* __restrict__ l, const T* __restrict__ m,
                                typename AccOf<T>::type* __restrict__ lse,
                                typename AccOf<T>::type* __restrict__ dsum, int64_t batch, int32_t v_d,
                                int32_t nq) {
  using A = typename AccOf<T>::type;
  const int64_t total = batch * nq;
  for (int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; i < total;
       i += int64_t(gridDim.x) * blockDim.x) {
    const int64_t b = i / nq, r = i - b * nq;
    A acc = A(0);
    const T* op = o + b * v_d * int64_t(nq) + r;
    const T* dp = d_o + b * v_d * int64_t(nq) + r;
    for (int c = 0; c < v_d; ++c) acc += to_acc<A>(op[int64_t(c) * nq]) * to_acc<A>(dp[int64_t(c) * nq]);
    dsum[i] = acc;
    const A lv = A(l[i]);
    const T mv = m[i];
    lse[i] = (lv > A(0) && !is_sentinel<T>(mv)) ? to_acc<A>(mv) + acc_log(lv) : -neg_inf<A>();
  }
}

// ---- backward dQ: one CTA per Q tile, streams K/V tiles ------------------------------------
// KC > 0 (wide): one CTA per (Q tile, slice of dQ's channels).
template <typename T, int BM, int BN, int NS, int KC = 0>
__global__ void __launch_bounds__(NT) bwd_dq_kernel(const BwdParams<T> p) {
  using A = typename AccOf<T>::type;
  constexpr int RM = BM / 16, CN = BN / 16;
  constexpr bool WIDE = KC > 0;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  A* Qs = reinterpret_cast<A*>(smem_raw);           // [d][BM]     (wide, streamed: [KC][BM])
  A* dOs = Qs + (WIDE && !p.res ? KC : p.d) * BM;   // [v_d][BM]   (wide, streamed: [KC][BM])
  A* Ks = dOs + (WIDE && !p.res ? KC : p.v_d) * BM; // [d][BN+1]   (wide: the K slice [sw][BN+1])  also dQ staging
  A* Vs = Ks + (WIDE ? p.sw : p.d) * (BN + 1);      // [v_d][BN+1] (wide: K and V chunks [KC][BN+1])
  A* Ds = Vs + (WIDE ? KC : p.v_d) * (BN + 1);      // [BM][BN+1]  dS tile

  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int rt = p.n_rtiles - 1 - int(blockIdx.x % p.n_rtiles);
  int64_t b = blockIdx.x / p.n_rtiles;
  int c_lo = 0, c_n = 0;  // wide: this CTA's dQ channels are c_lo .. c_lo + c_n - 1
  if constexpr (WIDE) {
    const int slice = int(b % p.n_sl);
    b /= p.n_sl;
    c_lo = slice * p.sw;
    c_n = min(p.sw, p.d - c_lo);
  }
  const int q0 = rt * BM;
  const int q_hi = min(q0 + BM, p.nq) - 1;
  const FaRule& rule = p.rule;
  const A scale = A(1) / sqrt(A(p.d));

  if (!WIDE || p.res) {
    load_tile<T, A>(Qs, p.q + b * p.d * int64_t(p.nq), p.d, BM, BM, p.nq, q0);
    load_tile<T, A>(dOs, p.d_o + b * p.v_d * int64_t(p.nq), p.v_d, BM, BM, p.nq, q0);
  }

  FaPos qpos[RM];
  A lse[RM], dsum[RM], dq[RM][NS];
#pragma unroll
  for (int i = 0; i < RM; ++i) {
    int qi = min(q0 + ty * RM + i, p.nq - 1);
    qpos[i] = fa_pos(rule, rule.q, qi);
    lse[i] = p.lse[b * p.nq + qi];
    dsum[i] = p.dsum[b * p.nq + qi];
#pragma unroll
    for (int s = 0; s < NS; ++s) dq[i][s] = A(0);
  }

  int kt_first, kt_last;
  fa_k_tile_range(rule, q0, q_hi, BN, &kt_first, &kt_last);
  for (int kt = kt_first; kt <= kt_last; ++kt) {
    const int k0 = kt * BN;
    const int k_hi = min(k0 + BN, p.nk) - 1;
    const int cls = fa_classify(rule, q0, q_hi, k0, k_hi);
    if (cls == FA_TILE_SKIP) continue;
    __syncthreads();
    A s[RM][CN], dp[RM][CN];
    if constexpr (!WIDE) {
      load_tile<T, A>(Ks, p.k + b * p.d * int64_t(p.nk), p.d, BN, BN + 1, p.nk, k0);
      load_tile<T, A>(Vs, p.v + b * p.v_d * int64_t(p.nk), p.v_d, BN, BN + 1, p.nk, k0);
      __syncthreads();
      gemm_s<A, BM, BN>(Qs, Ks, p.d, s, ty, tx);
      gemm_s<A, BM, BN>(dOs, Vs, p.v_d, dp, ty, tx);
    } else {
      load_tile<T, A>(Ks, p.k + (b * p.d + c_lo) * int64_t(p.nk), c_n, BN, BN + 1, p.nk, k0);
      gemm_s_chunked<T, A, BM, BN, KC>(Qs, p.res, p.q + b * p.d * int64_t(p.nq), p.nq, q0, Vs,
                                       p.k + b * p.d * int64_t(p.nk), p.nk, k0, p.d, s, ty, tx);
      gemm_s_chunked<T, A, BM, BN, KC>(dOs, p.res, p.d_o + b * p.v_d * int64_t(p.nq), p.nq, q0, Vs,
                                       p.v + b * p.v_d * int64_t(p.nk), p.nk, k0, p.v_d, dp, ty, tx);
    }
#pragma unroll
    for (int j = 0; j < CN; ++j) {
      const int kj = k0 + tx + 16 * j;
      const bool kvalid = kj < p.nk;
      const FaPos kpos = fa_pos(rule, rule.k, kvalid ? kj : p.nk - 1);
#pragma unroll
      for (int i = 0; i < RM; ++i) {
        bool ok = kvalid && (cls == FA_TILE_FULL || fa_attend(rule, qpos[i], kpos));
        A pr = ok ? acc_exp(s[i][j] * scale - lse[i]) : A(0);
        Ds[(ty * RM + i) * (BN + 1) + tx + 16 * j] = pr * (dp[i][j] - dsum[i]) * scale;
      }
    }
    __syncthreads();
    gemm_pv<A, BM, BN, NS>(Ds, Ks, WIDE ? c_n : p.d, dq, ty, tx);
  }
  __syncthreads();
  A* Os = Ks;  // [d][BM+1]  (wide: [c_n][BM+1])
#pragma unroll
  for (int i = 0; i < RM; ++i)
#pragma unroll
    for (int s = 0; s < NS; ++s) {
      int ch = tx + 16 * s;
      if (ch < (WIDE ? c_n : p.d)) Os[ch * (BM + 1) + ty * RM + i] = dq[i][s];
    }
  __syncthreads();
  T* og = p.d_q + (WIDE ? b * p.d + c_lo : b * p.d) * int64_t(p.nq);
  const int total = (WIDE ? c_n : p.d) * BM;
  for (int idx = threadIdx.x; idx < total; idx += NT) {
    int ch = idx / BM, r = idx - ch * BM;
    if (q0 + r < p.nq) og[int64_t(ch) * p.nq + q0 + r] = from_acc<T>(Os[ch * (BM + 1) + r]);
  }
}

// ---- backward dK/dV: one CTA per K tile (resident), streams Q/dO tiles ---------------------
// KC > 0 (wide): one CTA per (K tile, slice of the concatenated dK | dV channels). A slice lies in dK or in dV, never
// across both: a dV slice needs P only, a dK slice dS (and so dP = V . dO^T as well).
template <typename T, int BM, int BN, int NS, int KC = 0>
__global__ void __launch_bounds__(NT) bwd_dkdv_kernel(const BwdParams<T> p) {
  using A = typename AccOf<T>::type;
  constexpr int RM = BM / 16, CN = BN / 16;
  constexpr bool WIDE = KC > 0;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  A* Ks = reinterpret_cast<A*>(smem_raw);                     // [d][BM]     resident keys  (wide, streamed: [KC][BM])
  A* Vs = Ks + (WIDE && !p.res ? KC : p.d) * BM;              // [v_d][BM]   (wide, streamed: [KC][BM])
  A* Qs = Vs + (WIDE && !p.res ? KC : p.v_d) * BM;            // [d][BN+1]   streamed queries (also dK staging)
                                                              //   (wide: the Q or dO slice [max(sw, sw_v)][BN+1])
  A* dOs = Qs + (WIDE ? max(p.sw, p.sw_v) : p.d) * (BN + 1);  // [v_d][BN+1] (also dV staging)
                                                              //   (wide: Q and dO chunks [KC][BN+1])
  A* Ps = dOs + (WIDE ? KC : p.v_d) * (BN + 1);               // [BM][BN+1]  P^T
  A* Ds = Ps + BM * (BN + 1);                                 // [BM][BN+1]  dS^T
  A* lse_s = Ds + BM * (BN + 1);                              // [BN]
  A* dsum_s = lse_s + BN;                                     // [BN]

  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int rt = int(blockIdx.x % p.n_rtiles);  // early key tiles are the heavy ones under causal
  int64_t b = blockIdx.x / p.n_rtiles;
  int slice = 0;
  if constexpr (WIDE) {
    slice = int(b % p.n_sl);
    b /= p.n_sl;
  }
  const bool is_dk = !WIDE || slice < p.n_sl_k;      // wide: this CTA writes dK channels (else dV channels)
  const int c_lo = !WIDE ? 0 : is_dk ? slice * p.sw : (slice - p.n_sl_k) * p.sw_v;
  const int c_n = !WIDE ? 0 : is_dk ? min(p.sw, p.d - c_lo) : min(p.sw_v, p.v_d - c_lo);
  const int k0 = rt * BM;
  const int k_hi = min(k0 + BM, p.nk) - 1;
  const FaRule& rule = p.rule;
  const A scale = A(1) / sqrt(A(p.d));

  if (!WIDE || p.res) {
    load_tile<T, A>(Ks, p.k + b * p.d * int64_t(p.nk), p.d, BM, BM, p.nk, k0);
    load_tile<T, A>(Vs, p.v + b * p.v_d * int64_t(p.nk), p.v_d, BM, BM, p.nk, k0);
  }

  FaPos kpos[RM];
  bool kvalid[RM];
  A dk[RM][NS], dv[RM][NS];  // wide: dk is the slice's accumulator, dv is unused
#pragma unroll
  for (int i = 0; i < RM; ++i) {
    int ki = k0 + ty * RM + i;
    kvalid[i] = ki < p.nk;
    kpos[i] = fa_pos(rule, rule.k, min(ki, p.nk - 1));
#pragma unroll
    for (int s = 0; s < NS; ++s) dk[i][s] = dv[i][s] = A(0);
  }

  int qt_first, qt_last;
  fa_q_tile_range(rule, k0, k_hi, BN, &qt_first, &qt_last);
  for (int qt = qt_first; qt <= qt_last; ++qt) {
    const int q0 = qt * BN;
    const int q_hi = min(q0 + BN, p.nq) - 1;
    const int cls = fa_classify(rule, q0, q_hi, k0, k_hi);
    if (cls == FA_TILE_SKIP) continue;
    __syncthreads();
    if constexpr (!WIDE) {
      load_tile<T, A>(Qs, p.q + b * p.d * int64_t(p.nq), p.d, BN, BN + 1, p.nq, q0);
      load_tile<T, A>(dOs, p.d_o + b * p.v_d * int64_t(p.nq), p.v_d, BN, BN + 1, p.nq, q0);
    } else {
      const T* src = is_dk ? p.q + (b * p.d + c_lo) * int64_t(p.nq) : p.d_o + (b * p.v_d + c_lo) * int64_t(p.nq);
      load_tile<T, A>(Qs, src, c_n, BN, BN + 1, p.nq, q0);
    }
    if (threadIdx.x < BN) {
      int qi = q0 + threadIdx.x;
      bool v = qi < p.nq;
      lse_s[threadIdx.x] = v ? p.lse[b * p.nq + qi] : -neg_inf<A>();
      dsum_s[threadIdx.x] = v ? p.dsum[b * p.nq + qi] : A(0);
    }
    A st[RM][CN], dpt[RM][CN];
    if constexpr (!WIDE) {
      __syncthreads();
      gemm_s<A, BM, BN>(Ks, Qs, p.d, st, ty, tx);
      gemm_s<A, BM, BN>(Vs, dOs, p.v_d, dpt, ty, tx);
    } else {
      gemm_s_chunked<T, A, BM, BN, KC>(Ks, p.res, p.k + b * p.d * int64_t(p.nk), p.nk, k0, dOs,
                                       p.q + b * p.d * int64_t(p.nq), p.nq, q0, p.d, st, ty, tx);
      if (is_dk) {
        gemm_s_chunked<T, A, BM, BN, KC>(Vs, p.res, p.v + b * p.v_d * int64_t(p.nk), p.nk, k0, dOs,
                                         p.d_o + b * p.v_d * int64_t(p.nq), p.nq, q0, p.v_d, dpt, ty, tx);
      } else {
#pragma unroll
        for (int i = 0; i < RM; ++i)
#pragma unroll
          for (int j = 0; j < CN; ++j) dpt[i][j] = A(0);
      }
    }
#pragma unroll
    for (int j = 0; j < CN; ++j) {
      const int col = tx + 16 * j;
      const int qj = q0 + col;
      const bool qvalid = qj < p.nq;
      const FaPos qpos = fa_pos(rule, rule.q, qvalid ? qj : p.nq - 1);
      const A lse = lse_s[col], dsum = dsum_s[col];
#pragma unroll
      for (int i = 0; i < RM; ++i) {
        bool ok = qvalid && kvalid[i] && (cls == FA_TILE_FULL || fa_attend(rule, qpos, kpos[i]));
        A pr = ok ? acc_exp(st[i][j] * scale - lse) : A(0);
        Ps[(ty * RM + i) * (BN + 1) + col] = pr;
        Ds[(ty * RM + i) * (BN + 1) + col] = pr * (dpt[i][j] - dsum) * scale;
      }
    }
    __syncthreads();
    if constexpr (!WIDE) {
      gemm_pv<A, BM, BN, NS>(Ps, dOs, p.v_d, dv, ty, tx);
      gemm_pv<A, BM, BN, NS>(Ds, Qs, p.d, dk, ty, tx);
    } else {
      gemm_pv<A, BM, BN, NS>(is_dk ? Ds : Ps, Qs, c_n, dk, ty, tx);
    }
  }
  __syncthreads();
  if constexpr (WIDE) {
    A* Os = Qs;  // [c_n][BM+1]
#pragma unroll
    for (int i = 0; i < RM; ++i)
#pragma unroll
      for (int s = 0; s < NS; ++s) {
        int ch = tx + 16 * s;
        if (ch < c_n) Os[ch * (BM + 1) + ty * RM + i] = dk[i][s];
      }
    __syncthreads();
    T* og = is_dk ? p.d_k + (b * p.d + c_lo) * int64_t(p.nk) : p.d_v + (b * p.v_d + c_lo) * int64_t(p.nk);
    for (int idx = threadIdx.x; idx < c_n * BM; idx += NT) {
      int ch = idx / BM, r = idx - ch * BM;
      if (k0 + r < p.nk) og[int64_t(ch) * p.nk + k0 + r] = from_acc<T>(Os[ch * (BM + 1) + r]);
    }
    return;
  }
  A* Ok = Qs;   // [d][BM+1]
  A* Ov = dOs;  // [v_d][BM+1]
#pragma unroll
  for (int i = 0; i < RM; ++i)
#pragma unroll
    for (int s = 0; s < NS; ++s) {
      int ch = tx + 16 * s;
      if (ch < p.d) Ok[ch * (BM + 1) + ty * RM + i] = dk[i][s];
      if (ch < p.v_d) Ov[ch * (BM + 1) + ty * RM + i] = dv[i][s];
    }
  __syncthreads();
  T* gk = p.d_k + b * p.d * int64_t(p.nk);
  T* gv = p.d_v + b * p.v_d * int64_t(p.nk);
  for (int idx = threadIdx.x; idx < p.d * BM; idx += NT) {
    int ch = idx / BM, r = idx - ch * BM;
    if (k0 + r < p.nk) gk[int64_t(ch) * p.nk + k0 + r] = from_acc<T>(Ok[ch * (BM + 1) + r]);
  }
  for (int idx = threadIdx.x; idx < p.v_d * BM; idx += NT) {
    int ch = idx / BM, r = idx - ch * BM;
    if (k0 + r < p.nk) gv[int64_t(ch) * p.nk + k0 + r] = from_acc<T>(Ov[ch * (BM + 1) + r]);
  }
}

// ---- host-side launch helpers --------------------------------------------------------------
template <typename T>
static size_t fwd_smem(int d, int v_d, int BM) {
  using A = typename AccOf<T>::type;
  return sizeof(A) * (size_t(d) * BM + size_t(d) * (BM + 1) + size_t(v_d) * (BM + 1) + size_t(BM) * (BM + 1));
}
template <typename T>
static size_t dq_smem(int d, int v_d, int BM) {
  using A = typename AccOf<T>::type;
  return sizeof(A) * (size_t(d + v_d) * BM + size_t(d + v_d) * (BM + 1) + size_t(BM) * (BM + 1));
}
template <typename T>
static size_t dkdv_smem(int d, int v_d, int BM) {
  using A = typename AccOf<T>::type;
  return sizeof(A) * (size_t(d + v_d) * BM + size_t(d + v_d) * (BM + 1) + 2 * size_t(BM) * (BM + 1) + 2 * BM);
}

template <typename K, typename P>
static cudaError_t launch(const char* name, K kernel, const P& params, int64_t grid, size_t smem,
                          cudaStream_t stream) {
  cudaError_t e = plan::ensure_smem(kernel, int(smem));
  if (e != cudaSuccess) return e;
  ScopedKernel timed(name, stream);
  kernel<<<unsigned(grid), NT, smem, stream>>>(params);
  return cudaGetLastError();
}

constexpr size_t kSmemMax = 227 * 1024;

// Picks (BM, NS). Big tiles when channels <= 128, small tiles up to 256 channels.
template <typename T>
struct Tiles {
  static constexpr int kBig = sizeof(typename AccOf<T>::type) == 8 ? 32 : 64;
  static constexpr int kSmall = kBig / 2;
};

// ---- wide heads: more than 256 channels ------------------------------------------------------
// Each CTA owns a slice of at most 16 x NS <= 256 output channels, so the register accumulators keep the shape of the
// SMALL tiles; the grid is batch x row tiles x slices. Every slice recomputes S (and dP), so the host picks, among the
// instantiated NS, the slicing with the least arithmetic.
constexpr int kWideKC = 64;                 // channels per chunk of the streamed Q.K^T / dO.V^T reductions
constexpr int kWideNS[] = {4, 10, 16};   // instantiated accumulator widths (16 x NS channels per slice)

struct Slices {
  int n, w;  // n slices of w channels (a multiple of 16; the last slice may be narrower)
};
static Slices slices(int C, int ns) {
  const int u = (C + 15) / 16, n = (u + ns - 1) / ns;
  return {n, 16 * ((u + n - 1) / n)};
}

enum WideKind { kWideFwd, kWideDq, kWideDkdv };
struct WidePlan {
  int ns;
  Slices s, v;  // forward: O's channels; dQ: d; dK/dV: s = dK's channels, v = dV's channels
  bool res;     // the resident-side operands stay whole in shared memory
  size_t smem;
  int n_sl() const { return s.n + v.n; }
};

static WidePlan wide_plan(WideKind kind, int d, int v_d, int BM, size_t acc_bytes) {
  WidePlan best{};
  int64_t best_cost = -1;
  for (int ns : kWideNS) {
    WidePlan w{};
    w.ns = ns;
    int64_t cost;
    if (kind == kWideFwd) {
      w.s = slices(v_d, ns);
      cost = int64_t(w.s.n) * (d + 16 * ns);
    } else if (kind == kWideDq) {
      w.s = slices(d, ns);
      cost = int64_t(w.s.n) * (int64_t(d) + v_d + 16 * ns);
    } else {
      w.s = slices(d, ns);
      w.v = slices(v_d, ns);
      cost = int64_t(w.s.n) * (int64_t(d) + v_d + 16 * ns) + int64_t(w.v.n) * (d + 16 * ns);
    }
    if (best_cost < 0 || cost <= best_cost) {
      best = w;
      best_cost = cost;
    }
  }
  const size_t P = BM + 1, KC = kWideKC;
  const size_t res_rows = kind == kWideFwd ? size_t(d) : size_t(d) + v_d;
  const size_t chunk_rows = kind == kWideFwd ? KC : 2 * KC;
  const size_t other = kind == kWideFwd ? (KC + best.s.w + BM) * P
                       : kind == kWideDq ? (best.s.w + KC + BM) * P
                                         : (std::max(best.s.w, best.v.w) + KC + 2 * BM) * P + 2 * BM;
  const size_t resident = acc_bytes * (res_rows * BM + other);
  best.res = resident <= kSmemMax / 2;  // resident only where two CTAs still fit an SM
  best.smem = best.res ? resident : acc_bytes * (chunk_rows * BM + other);
  return best;
}

template <typename T>
static WidePlan wide_plan_t(WideKind kind, int d, int v_d) {
  return wide_plan(kind, d, v_d, Tiles<T>::kSmall, sizeof(typename AccOf<T>::type));
}

// batch x row tiles x slices of every launch of the call fits a 31-bit grid
template <typename T>
static bool wide_grid_fits(const LaunchArgs& a, bool backward) {
  constexpr int BM = Tiles<T>::kSmall;
  const int64_t rq = (int64_t(a.rule.q.total) + BM - 1) / BM, rk = (int64_t(a.rule.k.total) + BM - 1) / BM;
  auto fits = [&](int64_t tiles, const WidePlan& w) { return a.batch <= 0x7fffffffLL / std::max<int64_t>(1, tiles * w.n_sl()); };
  if (!backward) return fits(rq, wide_plan_t<T>(kWideFwd, a.d, a.v_d));
  return fits(rq, wide_plan_t<T>(kWideDq, a.d, a.v_d)) && fits(rk, wide_plan_t<T>(kWideDkdv, a.d, a.v_d));
}

template <typename T>
static cudaError_t forward_wide(FwdParams<T> p, cudaStream_t stream) {
  constexpr int BM = Tiles<T>::kSmall, KC = kWideKC;
  const WidePlan w = wide_plan_t<T>(kWideFwd, p.d, p.v_d);
  p.n_rtiles = (p.nq + BM - 1) / BM;
  p.sw = w.s.w;
  p.res = w.res;
  auto run = [&](int lo, int n) -> cudaError_t {
    p.slice_lo = lo;
    p.n_sl = n;
    const int64_t grid = p.batch * p.n_rtiles * n;
    switch (w.ns) {
      case 4: return launch("generic_fwd_wide", fwd_kernel<T, BM, BM, 4, KC>, p, grid, w.smem, stream);
      case 10: return launch("generic_fwd_wide", fwd_kernel<T, BM, BM, 10, KC>, p, grid, w.smem, stream);
      default: return launch("generic_fwd_wide", fwd_kernel<T, BM, BM, 16, KC>, p, grid, w.smem, stream);
    }
  };
  // accumulate = 1: every slice reads the incoming m and l, and slice 0 overwrites them, so slice 0 runs in a launch
  // of its own after the others
  if (p.accumulate && w.s.n > 1) {
    cudaError_t e = run(1, w.s.n - 1);
    if (e != cudaSuccess) return e;
    return run(0, 1);
  }
  return run(0, w.s.n);
}

template <typename T>
static cudaError_t backward_wide(BwdParams<T> p, cudaStream_t stream) {
  constexpr int BM = Tiles<T>::kSmall, KC = kWideKC;
  const WidePlan wq = wide_plan_t<T>(kWideDq, p.d, p.v_d);
  p.n_rtiles = (p.nq + BM - 1) / BM;
  p.sw = wq.s.w;
  p.n_sl = wq.n_sl();
  p.res = wq.res;
  int64_t grid = p.batch * p.n_rtiles * p.n_sl;
  cudaError_t e;
  switch (wq.ns) {
    case 4: e = launch("generic_bwd_dq_wide", bwd_dq_kernel<T, BM, BM, 4, KC>, p, grid, wq.smem, stream); break;
    case 10: e = launch("generic_bwd_dq_wide", bwd_dq_kernel<T, BM, BM, 10, KC>, p, grid, wq.smem, stream); break;
    default: e = launch("generic_bwd_dq_wide", bwd_dq_kernel<T, BM, BM, 16, KC>, p, grid, wq.smem, stream); break;
  }
  if (e != cudaSuccess) return e;
  const WidePlan wk = wide_plan_t<T>(kWideDkdv, p.d, p.v_d);
  p.n_rtiles = (p.nk + BM - 1) / BM;
  p.sw = wk.s.w;
  p.sw_v = wk.v.w;
  p.n_sl = wk.n_sl();
  p.n_sl_k = wk.s.n;
  p.res = wk.res;
  grid = p.batch * p.n_rtiles * p.n_sl;
  switch (wk.ns) {
    case 4: return launch("generic_bwd_dkdv_wide", bwd_dkdv_kernel<T, BM, BM, 4, KC>, p, grid, wk.smem, stream);
    case 10: return launch("generic_bwd_dkdv_wide", bwd_dkdv_kernel<T, BM, BM, 10, KC>, p, grid, wk.smem, stream);
    default: return launch("generic_bwd_dkdv_wide", bwd_dkdv_kernel<T, BM, BM, 16, KC>, p, grid, wk.smem, stream);
  }
}

template <typename T>
cudaError_t forward_t(const LaunchArgs& a, cudaStream_t stream) {
  FwdParams<T> p;
  p.q = (const T*)a.q; p.k = (const T*)a.k; p.v = (const T*)a.v;
  p.o = (T*)a.o; p.l = (typename LOf<T>::type*)a.l; p.m = (T*)a.m;
  p.d = a.d; p.v_d = a.v_d; p.nq = a.rule.q.total; p.nk = a.rule.k.total;
  p.batch = a.batch; p.accumulate = a.accumulate; p.rule = a.rule;
  if (std::max(a.d, a.v_d) > 256) return forward_wide<T>(p, stream);
  constexpr int BIG = Tiles<T>::kBig, SMALL = Tiles<T>::kSmall;
  const int ns = (a.v_d + 15) / 16;
#define FA_FWD(BM_, NS_)                                                                   \
  do {                                                                                     \
    p.n_rtiles = (p.nq + BM_ - 1) / BM_;                                                   \
    return launch("generic_fwd", fwd_kernel<T, BM_, BM_, NS_>, p, p.batch * p.n_rtiles,                   \
                  fwd_smem<T>(a.d, a.v_d, BM_), stream);                                   \
  } while (0)
  // fp64, up to 64 channels: 64 x 64 tiles (4 x 4 accumulators per thread: one shared-memory load per two DFMAs instead
  // of one per DFMA with the 32 x 32 tiles; C4 fp64 and the reference's fp64 benchmark shapes)
  if (sizeof(typename AccOf<T>::type) == 8 && ns <= 4 && a.d <= 64 && fwd_smem<T>(a.d, a.v_d, 64) <= kSmemMax)
    FA_FWD(64, 4);
  if (ns <= 2 && fwd_smem<T>(a.d, a.v_d, BIG) <= kSmemMax) FA_FWD(BIG, 2);
  if (ns <= 8 && fwd_smem<T>(a.d, a.v_d, BIG) <= kSmemMax) FA_FWD(BIG, 8);
  if (ns <= 16 && fwd_smem<T>(a.d, a.v_d, SMALL) <= kSmemMax) FA_FWD(SMALL, 16);
#undef FA_FWD
  return cudaErrorInvalidValue;
}

template <typename T>
cudaError_t backward_t(const LaunchArgs& a, cudaStream_t stream) {
  using A = typename AccOf<T>::type;
  BwdParams<T> p;
  p.q = (const T*)a.q; p.k = (const T*)a.k; p.v = (const T*)a.v; p.d_o = (const T*)a.d_o;
  p.d_q = (T*)a.d_q; p.d_k = (T*)a.d_k; p.d_v = (T*)a.d_v;
  p.d = a.d; p.v_d = a.v_d; p.nq = a.rule.q.total; p.nk = a.rule.k.total;
  p.batch = a.batch; p.rule = a.rule;
  A* lse = (A*)a.workspace;
  A* dsum = lse + p.batch * p.nq;
  p.lse = lse; p.dsum = dsum;
  {
    int64_t total = p.batch * p.nq;
    int blocks = int(std::min<int64_t>((total + 255) / 256, 148 * 8));
    cudaError_t e;
    {
      ScopedKernel timed("bwd_prep", stream);
      bwd_prep_kernel<T><<<blocks, 256, 0, stream>>>((const T*)a.o, (const T*)a.d_o,
                                                     (const typename LOf<T>::type*)a.l, (const T*)a.m,
                                                     lse, dsum, p.batch, p.v_d, p.nq);
      e = cudaGetLastError();
    }
    if (e != cudaSuccess) return e;
  }
  if (std::max(a.d, a.v_d) > 256) return backward_wide<T>(p, stream);
  constexpr int BIG = Tiles<T>::kBig, SMALL = Tiles<T>::kSmall;
  const int ns = (std::max(a.d, a.v_d) + 15) / 16;
#define FA_BWD(BM_, NS_)                                                                      \
  do {                                                                                        \
    p.n_rtiles = (p.nq + BM_ - 1) / BM_;                                                      \
    cudaError_t e = launch("generic_bwd_dq", bwd_dq_kernel<T, BM_, BM_, NS_>, p, p.batch * p.n_rtiles,          \
                           dq_smem<T>(a.d, a.v_d, BM_), stream);                              \
    if (e != cudaSuccess) return e;                                                           \
    p.n_rtiles = (p.nk + BM_ - 1) / BM_;                                                      \
    return launch("generic_bwd_dkdv", bwd_dkdv_kernel<T, BM_, BM_, NS_>, p, p.batch * p.n_rtiles,                 \
                  dkdv_smem<T>(a.d, a.v_d, BM_), stream);                                     \
  } while (0)
  if (sizeof(A) == 8 && ns <= 4 && dkdv_smem<T>(a.d, a.v_d, 64) <= kSmemMax) FA_BWD(64, 4);
  if (ns <= 2 && dkdv_smem<T>(a.d, a.v_d, BIG) <= kSmemMax) FA_BWD(BIG, 2);
  if (ns <= 8 && dkdv_smem<T>(a.d, a.v_d, BIG) <= kSmemMax) FA_BWD(BIG, 8);
  if (ns <= 16 && dkdv_smem<T>(a.d, a.v_d, SMALL) <= kSmemMax) FA_BWD(SMALL, 16);
#undef FA_BWD
  return cudaErrorInvalidValue;
}

}  // namespace generic

bool generic_supports(const LaunchArgs& a, bool backward) {
  if (a.layout != 0) return false;
  if (a.d <= 256 && a.v_d <= 256) return true;
  switch (a.dtype) {
    case 0: return generic::wide_grid_fits<__half>(a, backward);
    case 3: return generic::wide_grid_fits<__nv_bfloat16>(a, backward);
    case 1: return generic::wide_grid_fits<float>(a, backward);
    default: return generic::wide_grid_fits<double>(a, backward);
  }
}

size_t generic_workspace_bytes(int dtype, int64_t batch, int64_t nq, bool backward) {
  if (!backward) return 0;
  return size_t(2) * size_t(batch) * size_t(nq) * (dtype == 2 ? 8 : 4);
}

cudaError_t generic_forward(const LaunchArgs& a, cudaStream_t stream) {
  switch (a.dtype) {
    case 0: return generic::forward_t<__half>(a, stream);
    case 3: return generic::forward_t<__nv_bfloat16>(a, stream);
    case 1: return generic::forward_t<float>(a, stream);
    default: return generic::forward_t<double>(a, stream);
  }
}

cudaError_t generic_backward(const LaunchArgs& a, cudaStream_t stream) {
  switch (a.dtype) {
    case 0: return generic::backward_t<__half>(a, stream);
    case 3: return generic::backward_t<__nv_bfloat16>(a, stream);
    case 1: return generic::backward_t<float>(a, stream);
    default: return generic::backward_t<double>(a, stream);
  }
}

}  // namespace fa
