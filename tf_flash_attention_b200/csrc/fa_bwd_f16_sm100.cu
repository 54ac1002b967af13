// fa_bwd_f16_sm100.cu — Blackwell-native 16-bit (fp16 / bf16) backward: two tcgen05/TMEM/TMA kernels.
// Every kernel takes the element type T (__half or __nv_bfloat16) of Q, K, V, O, m, dO and the gradients, which is also
// the type P and dS are handed to the tensor cores in.
//
// Replaces the reference's BackwardImpl (flash_attention/kernel/flash_attention.cu:1079-1967), which
// keeps a K/V tile per CTA, loops over Q tiles under a global spin lock and read-modify-writes dQ in
// HBM with scalar FMAs. Here the work is split so that no inter-CTA communication is needed:
//
//   bwd_dq_kernel   : CTA = 2 x 128 query rows (ping-pong), streams 64-key K/V tiles
//        S  = Q K^T        (SS, both operands MN-major straight from the channel-first layout)
//        dP = dO V^T       (SS, MN-major)
//        dS = P o (dP - D) , P = exp2(S*scale*log2e - LSE2)      (softmax warps, TMEM -> regs -> TMEM)
//        dQ += dS K        (TS: dS from TMEM, K tile re-read K-major)
//   bwd_dkdv_kernel : CTA = 128 keys, streams 64-query Q/dO tiles into two ping-pong slots
//        S^T = K Q^T, dP^T = V dO^T  (SS, MN-major)
//        dV += P^T dO, dK += dS^T Q  (TS: P^T / dS^T from TMEM; dO / Q tiles re-read K-major)
//   bwd_fused_kernel (head_dim 128): bwd_dkdv_kernel + dQ^T = K^T dS^T in the same pass, dQ accumulated
//        across key tiles with TMA reduce-add into an fp32 scratch tensor (see its header comment)
// Formulas as in the reference: P = exp(s*scale - m)/l (flash_attention.cu:1838-1841),
// dS = P (dP - D) scale (:1544-1546), D = rowsum(dO o O) (:1882-1891).
#include "fa_common.cuh"
#include "fa_launch.h"
#include "fa_plan.h"
#include "sm100_ptx.cuh"
#include "sm100_tiles.cuh"

#include <cudaTypedefs.h>

#include <type_traits>

namespace fa {
namespace sm100 {

using namespace ptx;

bool make_map_2d(CUtensorMap* map, const void* base, int64_t rows, int64_t cols, int box_cols, int box_rows,
                 bool swizzle128);  // fa_fwd_f16_sm100.cu
bool make_map_3d(CUtensorMap* map, const void* base, int64_t batch, int64_t channels, int64_t seq, int64_t pitch,
                 int box_rows, bool swizzle128, CUtensorMapDataType dtype);  // fa_fwd_f16_sm100.cu
bool make_map_cl(CUtensorMap* map, const void* base, int64_t outer, int64_t heads, int64_t channels, int64_t seq,
                 int box_rows, CUtensorMapDataType dtype);  // fa_fwd_f16_sm100.cu

// Workspace of the fp16 backward: [LSE2, D (+ pad)] [fp32 dQ scratch of the fused head_dim-128 kernel] [pitch-padded
// copies of the q-length / k-length tensors when their length is not a multiple of 8 (fa_pack.cu)].
struct BwdLayout {
  bool pack_q, pack_k;
  size_t off_acc, off_q, off_do, off_dq, off_k, off_v, off_dk, off_dv, total;
};
BwdLayout bwd_layout(const LaunchArgs& a);

constexpr int kBM = 128;        // rows owned by one softmax warpgroup (TMEM lanes)
constexpr int kBN = 64;         // streamed tile width
constexpr int kBwdThreads = 384;
constexpr float kLog2eB = 1.4426950408889634f;
constexpr int kStatPad = 64;    // padding (floats) behind the LSE2 / D arrays for the bulk copies

// dS enters the tensor cores as fp16. |dS| = P |dP - D| reaches several units on rows that attend few keys, where one
// fp16 rounding (relative 2^-11) is already ~1e-3 absolute, and dK / dQ sum such terms. With SPLIT the softmax warps
// hand over dS as a hi + lo pair of fp16 values (lo = fp16(dS - hi), written into the TMEM columns the packed hi half
// leaves free) and the products dQ = dS K, dK = dS^T Q are issued twice, so dS carries ~22 mantissa bits (bf16: the
// same pair of bf16 values, ~16 bits).
template <typename T> __device__ __forceinline__ void split2(float a, float b, uint32_t& hi, uint32_t& lo);
template <> __device__ __forceinline__ void split2<__half>(float a, float b, uint32_t& hi, uint32_t& lo) {
  const __half2 h = __floats2half2_rn(a, b);
  const float2 f = __half22float2(h);
  const __half2 l = __floats2half2_rn(a - f.x, b - f.y);
  hi = *reinterpret_cast<const uint32_t*>(&h);
  lo = *reinterpret_cast<const uint32_t*>(&l);
}
template <> __device__ __forceinline__ void split2<__nv_bfloat16>(float a, float b, uint32_t& hi, uint32_t& lo) {
  hi = pack2<__nv_bfloat16>(a, b);
  lo = pack2<__nv_bfloat16>(a - __uint_as_float(hi << 16), b - __uint_as_float(hi & 0xffff0000u));
}

struct alignas(64) BwdParams {
  CUtensorMap map_q, map_k, map_v, map_do;   // SW128 loads, box 64 x channels
  CUtensorMap map_dq, map_dk, map_dv;        // plain stores, box 64 x channels
  FaRule rule;
  const float* lse2;   // [batch*nq + pad]  (m + log l) * log2(e), +inf on empty rows
  const float* dsum;   // [batch*nq + pad]  rowsum(dO o O)
  int32_t nq, nk, n_blocks, batch;
  int32_t heads;       // channel-last tensors: batch element = outer * heads + head
  int32_t stat_pitch;  // floats per batch element in lse2 / dsum: nq rounded up to 4 (16-byte rows for the bulk copies)
  int32_t exact_d;     // split-operand dQ kernel: replace D = rowsum(dO o O) (O is fp16-rounded) by rowsum(P o dP)
  float* dsum_out;     // where that kernel leaves the exact D for the dK/dV kernel launched behind it (== dsum)
  float scale_log2, scale;
};

// ---- preprocess: LSE2 and D -------------------------------------------------------------------
template <typename T>
__global__ void bwd_prep_f16(const T* __restrict__ o, const T* __restrict__ d_o,
                             const float* __restrict__ l, const T* __restrict__ m, float* __restrict__ lse2,
                             float* __restrict__ dsum, int64_t batch, int32_t v_d, int32_t nq, int32_t sp) {
  const int64_t total = batch * sp;
  // the padding behind both arrays (and behind each batch element's row when nq is not a multiple of 4) is read by the
  // 64-wide bulk copies of the last, ragged query tile: keep it finite (a NaN there would turn the masked
  // 0 * (dP - D) into NaN)
  if (blockIdx.x == gridDim.x - 1 && threadIdx.x < kStatPad) {
    lse2[total + threadIdx.x] = __int_as_float(0x7f800000);
    dsum[total + threadIdx.x] = 0.f;
  }
  // two adjacent query positions per thread -> pair loads, coalesced along the sequence (nq and sp are even here)
  for (int64_t i2 = (blockIdx.x * int64_t(blockDim.x) + threadIdx.x) * 2; i2 < total;
       i2 += int64_t(gridDim.x) * blockDim.x * 2) {
    const int64_t b = i2 / sp, r = i2 - b * sp;
    if (r >= nq) {
      lse2[i2] = lse2[i2 + 1] = __int_as_float(0x7f800000);
      dsum[i2] = dsum[i2 + 1] = 0.f;
      continue;
    }
    const Pair<T>* op = reinterpret_cast<const Pair<T>*>(o + b * v_d * int64_t(nq) + r);
    const Pair<T>* dp = reinterpret_cast<const Pair<T>*>(d_o + b * v_d * int64_t(nq) + r);
    float a0 = 0.f, a1 = 0.f;
    const int64_t pitch2 = nq / 2;
#pragma unroll 4
    for (int c = 0; c < v_d; ++c) {
      const float2 x = to_float2(op[c * pitch2]);
      const float2 y = to_float2(dp[c * pitch2]);
      a0 = fmaf(x.x, y.x, a0);
      a1 = fmaf(x.y, y.y, a1);
    }
    dsum[i2] = a0;
    dsum[i2 + 1] = a1;
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      const float lv = l[b * nq + r + e];
      const T mv = m[b * nq + r + e];
      lse2[i2 + e] = (lv > 0.f && !is_sentinel<T>(mv)) ? (to_acc<float>(mv) + logf(lv)) * kLog2eB
                                                             : __int_as_float(0x7f800000);
    }
  }
}

// any query length (odd included): one thread per query position, scalar loads coalesced along the sequence
template <typename T>
__global__ void bwd_prep_f16_any(const T* __restrict__ o, const T* __restrict__ d_o,
                                 const float* __restrict__ l, const T* __restrict__ m, float* __restrict__ lse2,
                                 float* __restrict__ dsum, int64_t batch, int32_t v_d, int32_t nq, int32_t sp) {
  const int64_t total = batch * sp;
  if (blockIdx.x == gridDim.x - 1 && threadIdx.x < kStatPad) {
    lse2[total + threadIdx.x] = __int_as_float(0x7f800000);
    dsum[total + threadIdx.x] = 0.f;
  }
  for (int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; i < total; i += int64_t(gridDim.x) * blockDim.x) {
    const int64_t b = i / sp, r = i - b * sp;
    if (r >= nq) {
      lse2[i] = __int_as_float(0x7f800000);
      dsum[i] = 0.f;
      continue;
    }
    const T* op = o + b * v_d * int64_t(nq) + r;
    const T* dp = d_o + b * v_d * int64_t(nq) + r;
    float acc = 0.f;
#pragma unroll 4
    for (int c = 0; c < v_d; ++c) acc = fmaf(to_acc<float>(op[c * int64_t(nq)]), to_acc<float>(dp[c * int64_t(nq)]), acc);
    dsum[i] = acc;
    const float lv = l[b * nq + r];
    const T mv = m[b * nq + r];
    lse2[i] = (lv > 0.f && !is_sentinel<T>(mv)) ? (to_acc<float>(mv) + logf(lv)) * kLog2eB
                                                      : __int_as_float(0x7f800000);
  }
}

// channel-last O / dO ([outer][q][heads][v_d], v_d a multiple of 8): a group of G lanes (the power of two >= v_d / 8)
// reads one row's channels as 16-byte chunks and reduces with shuffles; one thread per (outer, q, head) row would touch
// 16 bytes of every 2 * v_d-byte row per instruction
template <typename T, int G>
__global__ void bwd_prep_f16_cl(const T* __restrict__ o, const T* __restrict__ d_o,
                                const float* __restrict__ l, const T* __restrict__ m, float* __restrict__ lse2,
                                float* __restrict__ dsum, int64_t outer, int32_t heads, int32_t v_d, int32_t nq,
                                int32_t sp) {
  const int64_t batch = outer * heads, total = batch * sp;
  if (blockIdx.x == gridDim.x - 1 && threadIdx.x < kStatPad) {
    lse2[total + threadIdx.x] = __int_as_float(0x7f800000);
    dsum[total + threadIdx.x] = 0.f;
  }
  // the padding behind each batch element's row (nq not a multiple of 4)
  for (int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; i < batch * (sp - nq);
       i += int64_t(gridDim.x) * blockDim.x) {
    const int64_t b = i / (sp - nq), r = nq + i % (sp - nq);
    lse2[b * sp + r] = __int_as_float(0x7f800000);
    dsum[b * sp + r] = 0.f;
  }
  const int g = threadIdx.x % G;
  const int64_t rows = outer * nq * heads;
  // every lane of a warp runs the same number of iterations (the shuffles below name the whole warp): rows past the end
  // are predicated off, not skipped
  const int64_t first = (blockIdx.x * int64_t(blockDim.x) + threadIdx.x) / G, step = int64_t(gridDim.x) * blockDim.x / G;
  const int64_t warp_first = (blockIdx.x * int64_t(blockDim.x) + (threadIdx.x & ~31)) / G;
  for (int64_t it = 0; warp_first + it * step < rows; ++it) {
    const int64_t row = first + it * step;
    const bool live = row < rows;
    float acc = 0.f;
    if (live && g * 8 < v_d) {
      const uint4 x = *reinterpret_cast<const uint4*>(o + row * v_d + g * 8);
      const uint4 y = *reinterpret_cast<const uint4*>(d_o + row * v_d + g * 8);
      const Pair<T>* xh = reinterpret_cast<const Pair<T>*>(&x);
      const Pair<T>* yh = reinterpret_cast<const Pair<T>*>(&y);
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const float2 a = to_float2(xh[e]), c = to_float2(yh[e]);
        acc = fmaf(a.x, c.x, acc);
        acc = fmaf(a.y, c.y, acc);
      }
    }
#pragma unroll
    for (int w = G / 2; w > 0; w >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, w, G);
    if (live && g == 0) {
      const int64_t h = row % heads, oq = row / heads, q = oq % nq, ob = oq / nq;
      const int64_t b = ob * heads + h;
      dsum[b * sp + q] = acc;
      const float lv = l[b * nq + q];
      const T mv = m[b * nq + q];
      lse2[b * sp + q] = (lv > 0.f && !is_sentinel<T>(mv)) ? (to_acc<float>(mv) + logf(lv)) * kLog2eB
                                                                 : __int_as_float(0x7f800000);
    }
  }
}

// =================================================================================================
// dQ kernel
// =================================================================================================
template <int D, int VD>
struct DqCfg {
  static constexpr int kStages = 3;
  static constexpr int kQBytes = kBM * D * 2;       // also the dQ staging tile
  static constexpr int kDoBytes = kBM * VD * 2;
  static constexpr int kKBytes = kBN * D * 2;
  static constexpr int kVBytes = kBN * VD * 2;
  static constexpr int kStageBytes = kKBytes + kVBytes;
  static constexpr int kRingOffset = 2 * (kQBytes + kDoBytes);
  static constexpr int kBarOffset = kRingOffset + kStages * kStageBytes;
  static constexpr int kNumBars = 2 + 2 * kStages + 2 + 2 + 2;
  static constexpr int kSchedOffset = kBarOffset + kNumBars * 8 + 16;
  static constexpr int kSmemBytes = kSchedOffset + int(sizeof(TileSchedule)) + 1024;
};

template <typename T, int D, int VD, bool SPLIT, bool CL>
__global__ void __launch_bounds__(kBwdThreads, 1) bwd_dq_kernel(const __grid_constant__ BwdParams p) {
  using Cfg = DqCfg<D, VD>;
  constexpr int kStages = Cfg::kStages;
  // precise gradients with the exact row sum D = rowsum(P o dP) (see bwd_dq_small_kernel): needs a second accumulator
  // A2 = P K per Q tile, which fits behind dQ_i only while D <= 64
  constexpr bool kExact = SPLIT && D <= 64;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  const uint32_t q_smem = smem_base;                       // [2][kQBytes]
  const uint32_t do_smem = smem_base + 2 * Cfg::kQBytes;   // [2][kDoBytes]
  const uint32_t ring = smem_base + Cfg::kRingOffset;
  const uint32_t bars = smem_base + Cfg::kBarOffset;
  const uint32_t bar_q_full = bars;
  const uint32_t bar_kv_full = bars + 16;
  const uint32_t bar_kv_empty = bar_kv_full + 8 * kStages;
  const uint32_t bar_s_full = bar_kv_empty + 8 * kStages;
  const uint32_t bar_p_ready = bar_s_full + 16;
  const uint32_t bar_final = bar_p_ready + 16;
  const uint32_t tmem_slot = bar_final + 16;
  volatile uint32_t* tmem_slot_gen =
      reinterpret_cast<volatile uint32_t*>(smem_gen + Cfg::kBarOffset + Cfg::kNumBars * 8);

  const int warp = threadIdx.x >> 5;
  const FaRule& rule = p.rule;
  const int b = int(blockIdx.x / p.n_blocks);                     // head-major: K/V stay in L2
  const BatchCoord bc = batch_coord<CL>(b, p.heads);
  const int pair = p.n_blocks - 1 - int(blockIdx.x % p.n_blocks);  // heavy (late) rows first
  const int q0 = pair * (2 * kBM);
  const int q_hi = min(q0 + 2 * kBM, p.nq) - 1;
  int kt_first, kt_last;
  fa_k_tile_range(rule, q0, q_hi, kBN, &kt_first, &kt_last);
  TileSchedule* sched = reinterpret_cast<TileSchedule*>(smem_gen + Cfg::kSchedOffset);
  {
    const int lo[2] = {q0, q0 + kBM};
    const int hi[2] = {min(q0 + kBM, p.nq) - 1, min(q0 + 2 * kBM, p.nq) - 1};
    const bool valid[2] = {q0 < p.nq, q0 + kBM < p.nq};
    build_schedule(sched, rule, true, lo, hi, valid, 2, kt_first, kt_last, kBN, p.nk, kBwdThreads / 32);
  }

  if (warp == 8) {
    if (elect_one()) {
      prefetch_tensormap(&p.map_q);
      prefetch_tensormap(&p.map_k);
      prefetch_tensormap(&p.map_v);
      prefetch_tensormap(&p.map_do);
      prefetch_tensormap(&p.map_dq);
    }
  } else if (warp == 9) {
    if (elect_one()) {
      for (int i = 0; i < 2; ++i) {
        mbar_init(bar_q_full + 8 * i, 1);
        mbar_init(bar_s_full + 8 * i, 1);
        mbar_init(bar_p_ready + 8 * i, kBM);
        mbar_init(bar_final + 8 * i, 1);
      }
      for (int s = 0; s < kStages; ++s) {
        mbar_init(bar_kv_full + 8 * s, 1);
        mbar_init(bar_kv_empty + 8 * s, 1);
      }
      fence_barrier_init();
    }
  } else if (warp == 10) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_gen;
  // TMEM columns: S_i [i*64, +64)  dP_i [128+i*64, +64)  dQ_i [256+i*128, +D)

  if (warp >= 8) {
    setmaxnreg_dec<56>();
    if (warp == 8) {
      if (elect_one()) {
        for (int i = 0; i < 2; ++i) {
          mbar_arrive_expect_tx(bar_q_full + 8 * i, Cfg::kQBytes + Cfg::kDoBytes);
          tile_load<CL>(q_smem + i * Cfg::kQBytes, &p.map_q, bar_q_full + 8 * i, q0 + i * kBM, kBM, D, bc);
          tile_load<CL>(do_smem + i * Cfg::kDoBytes, &p.map_do, bar_q_full + 8 * i, q0 + i * kBM, kBM, VD, bc);
        }
        int t = 0;
        TileIter it;
        it.init(sched, 2, kt_first, kt_last);
        int kt, tw, tb;
        while (it.next(&kt, &tw, &tb)) {
          const int s = t % kStages, u = t / kStages;
          mbar_wait(bar_kv_empty + 8 * s, (u & 1) ^ 1);
          mbar_arrive_expect_tx(bar_kv_full + 8 * s, Cfg::kStageBytes);
          tile_load<CL>(ring + s * Cfg::kStageBytes, &p.map_k, bar_kv_full + 8 * s, kt * kBN, kBN, D, bc);
          tile_load<CL>(ring + s * Cfg::kStageBytes + Cfg::kKBytes, &p.map_v, bar_kv_full + 8 * s, kt * kBN, kBN, VD, bc);
          ++t;
        }
      }
    } else if (warp == 9) {
      if (elect_one()) {
        TileIter it;
        it.init(sched, 2, kt_first, kt_last);
        const int n = it.count();
        constexpr uint32_t idesc_s = idesc_16<T>(kBM, kBN, tile_mn_major<CL>(true), tile_mn_major<CL>(true));
        constexpr uint32_t idesc_dq = idesc_16<T>(kBM, D, false, tile_mn_major<CL>(false));
        auto issue_s_dp = [&](int i, int stage) {
          const uint32_t k_s = ring + stage * Cfg::kStageBytes, v_s = k_s + Cfg::kKBytes;
#pragma unroll
          for (int ks = 0; ks < D / 16; ++ks)
            mma_ss(tmem_base + i * kBN, tile_desc<CL>(q_smem + i * Cfg::kQBytes, ks, kBM, D, true),
                   tile_desc<CL>(k_s, ks, kBN, D, true), idesc_s, ks > 0);
#pragma unroll
          for (int ks = 0; ks < VD / 16; ++ks)
            mma_ss(tmem_base + 128 + i * kBN,
                   tile_desc<CL>(do_smem + i * Cfg::kDoBytes, ks, kBM, VD, true),
                   tile_desc<CL>(v_s, ks, kBN, VD, true), idesc_s, ks > 0);
        };
        auto issue_dq = [&](int i, int stage, bool accumulate) {
          const uint32_t k_s = ring + stage * Cfg::kStageBytes;
#pragma unroll
          for (int ks = 0; ks < kBN / 16; ++ks)
            mma_ts(tmem_base + 256 + i * 128, tmem_base + i * kBN + ks * 8,
                   tile_desc<CL>(k_s, ks, kBN, D, false), idesc_dq, (accumulate || ks > 0) ? 1u : 0u);
          if constexpr (SPLIT) {   // dS lo halves: the 32 columns behind the packed hi halves
#pragma unroll
            for (int ks = 0; ks < kBN / 16; ++ks)
              mma_ts(tmem_base + 256 + i * 128, tmem_base + i * kBN + 32 + ks * 8,
                     tile_desc<CL>(k_s, ks, kBN, D, false), idesc_dq, 1u);
          }
          if constexpr (kExact) {   // A2_i += P K: P (fp16) in the dP columns, A2 in the upper half of the dQ_i columns
#pragma unroll
            for (int ks = 0; ks < kBN / 16; ++ks)
              mma_ts(tmem_base + 256 + i * 128 + 64, tmem_base + 128 + i * kBN + ks * 8,
                     tile_desc<CL>(k_s, ks, kBN, D, false), idesc_dq, (accumulate || ks > 0) ? 1u : 0u);
          }
        };
        if (n > 0) {
          mbar_wait(bar_kv_full + 0, 0);
          for (int i = 0; i < 2; ++i) {
            mbar_wait(bar_q_full + 8 * i, 0);
            tc_fence_after();
            issue_s_dp(i, 0);
            mma_commit(bar_s_full + 8 * i);
          }
          for (int j = 0; j < n; ++j) {
            const int sj = j % kStages, sn = (j + 1) % kStages;
            for (int i = 0; i < 2; ++i) {
              mbar_wait(bar_p_ready + 8 * i, j & 1);
              tc_fence_after();
              issue_dq(i, sj, j > 0);
              if (i == 1) mma_commit(bar_kv_empty + 8 * sj);
              if (j + 1 < n) {
                if (i == 0) {
                  mbar_wait(bar_kv_full + 8 * sn, ((j + 1) / kStages) & 1);
                  tc_fence_after();
                }
                issue_s_dp(i, sn);
                mma_commit(bar_s_full + 8 * i);
              } else {
                mma_commit(bar_final + 8 * i);
              }
            }
          }
        }
      }
    }
  } else {
    setmaxnreg_inc<224>();
    const int i = warp >> 2;
    const int r = threadIdx.x & 127;
    const uint32_t lane_addr = uint32_t((warp & 3) * 32) << 16;
    const uint32_t t_s = tmem_base + lane_addr + i * kBN;
    const uint32_t t_dp = tmem_base + lane_addr + 128 + i * kBN;
    const uint32_t t_dq = tmem_base + lane_addr + 256 + i * 128;
    const int tq0 = q0 + i * kBM;
    const int tq_hi = min(tq0 + kBM, p.nq) - 1;
    const bool tile_valid = tq0 < p.nq;
    const int qi = tq0 + r;
    const bool q_valid = qi < p.nq;
    const FaPos qpos = fa_pos(rule, rule.q, min(qi, p.nq - 1));
    const float lse2 = q_valid ? p.lse2[int64_t(b) * p.stat_pitch + qi] : __int_as_float(0x7f800000);
    const float dsum = q_valid ? p.dsum[int64_t(b) * p.stat_pitch + qi] : 0.f;
    const float scale_log2 = p.scale_log2;
    float d_exact = 0.f;   // kExact: rowsum(P o dP) of this thread's row
    int j = 0;
    TileIter it;
    it.init(sched, 2, kt_first, kt_last);
    int kt, tw, tb;
    while (it.next(&kt, &tw, &tb)) {
      const int k0 = kt * kBN;
      const int k_hi = min(k0 + kBN, p.nk) - 1;
      const int cls = it.cls(i, tw, tb);
      const bool ragged = k0 + kBN > p.nk;
      mbar_wait(bar_s_full + 8 * i, j & 1);
      tc_fence_after();
      // masks first: nothing that may move registers between tcgen05.ld and tcgen05.wait::ld
      uint32_t okmask_lo = 0xffffffffu, okmask_hi = 0xffffffffu;
      if (cls == FA_TILE_SKIP) {
        okmask_lo = okmask_hi = 0u;
      } else if (cls == FA_TILE_PARTIAL || ragged) {
        const int nvalid = k_hi - k0 + 1;
        if (rule.dims == 1 && rule.rule != 2) {
          int lo, hi;
          interval_1d(rule, true, qpos, k0, nvalid, &lo, &hi);
          okmask_lo = interval_bits32(lo, hi, 0);
          okmask_hi = interval_bits32(lo, hi, 32);
        } else {
          okmask_lo = tile_mask32(rule, true, qpos, k0, 0, nvalid);
          okmask_hi = tile_mask32(rule, true, qpos, k0, 32, nvalid);
        }
      }
      float s[64], dp[64];
      tmem_ld32f(t_s, &s[0]);
      tmem_ld32f(t_s + 32, &s[32]);
      tmem_ld32f(t_dp, &dp[0]);
      tmem_ld32f(t_dp + 32, &dp[32]);
      tmem_wait_ld();
      uint32_t pk[32], pl[SPLIT ? 32 : 1], pp[kExact ? 32 : 1];
#pragma unroll
      for (int c = 0; c < 64; c += 2) {
        const uint32_t mword = c < 32 ? okmask_lo : okmask_hi;
        float p0 = ex2(fmaf(s[c], scale_log2, -lse2));
        float p1 = ex2(fmaf(s[c + 1], scale_log2, -lse2));
        p0 = (mword >> (c & 31)) & 1u ? p0 : 0.f;
        p1 = (mword >> ((c + 1) & 31)) & 1u ? p1 : 0.f;
        if constexpr (kExact) {
          d_exact = fmaf(p0, dp[c], d_exact);
          d_exact = fmaf(p1, dp[c + 1], d_exact);
          pp[c >> 1] = pack2<T>(p0, p1);
        }
        if constexpr (SPLIT)
          split2<T>(p0 * (dp[c] - dsum), p1 * (dp[c + 1] - dsum), pk[c >> 1], pl[c >> 1]);
        else
          pk[c >> 1] = pack2<T>(p0 * (dp[c] - dsum), p1 * (dp[c + 1] - dsum));
      }
      tmem_st32(t_s, pk);
      if constexpr (SPLIT) tmem_st32(t_s + 32, pl);
      if constexpr (kExact) tmem_st32(t_dp, pp);
      tmem_wait_st();
      tc_fence_before();
      mbar_arrive(bar_p_ready + 8 * i);
      ++j;
    }
    // epilogue: dQ = scale * acc -> fp16 -> smem [D][64] x2 -> TMA store
    uint8_t* stage_gen = smem_gen + i * Cfg::kQBytes;
    if (j > 0) {
      mbar_wait(bar_final + 8 * i, 0);
      tc_fence_after();
      float delta = 0.f;
      if constexpr (kExact) {
        if (p.exact_d) {
          delta = d_exact - dsum;
          if (q_valid) p.dsum_out[int64_t(b) * p.stat_pitch + qi] = d_exact;
        }
      }
#pragma unroll
      for (int c = 0; c < D / 32; ++c) {
        float o[32];
        tmem_ld32f(t_dq + c * 32, o);
        tmem_wait_ld();
        if constexpr (kExact) {
          float o2[32];
          tmem_ld32f(t_dq + 64 + c * 32, o2);
          tmem_wait_ld();
#pragma unroll
          for (int e = 0; e < 32; ++e) o[e] = fmaf(-delta, o2[e], o[e]);
        }
        stage_row32<CL, T>(stage_gen, r, c * 32, kBM, D, o, p.scale);
      }
    } else {
      mbar_wait(bar_q_full + 8 * i, 0);
      stage_row_zero<CL>(stage_gen, r, 0, D, kBM, D);
    }
    fence_proxy_async_smem();
    named_bar_sync(1 + i, kBM);
    if (r == 0 && tile_valid) {
      tile_store<CL>(&p.map_dq, q_smem + i * Cfg::kQBytes, tq0, kBM, D, p.nq, bc);
      tma_store_commit();
      tma_store_wait_read();
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 10) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// =================================================================================================
// dQ kernel, small configuration (head_dim 64): one 128-row Q tile per CTA, one S / dP slot, both softmax
// warpgroups split the 64 key columns, 256 TMEM columns and ~82 KB of shared memory -> two CTAs per SM
// =================================================================================================
template <int D, int VD>
struct DqSmallCfg {
  static constexpr int kStages = 3;
  static constexpr int kQBytes = kBM * D * 2;       // also the dQ staging tile
  static constexpr int kDoBytes = kBM * VD * 2;
  static constexpr int kKBytes = kBN * D * 2;
  static constexpr int kVBytes = kBN * VD * 2;
  static constexpr int kStageBytes = kKBytes + kVBytes;
  static constexpr int kRingOffset = kQBytes + kDoBytes;
  static constexpr int kBarOffset = kRingOffset + kStages * kStageBytes;
  static constexpr int kNumBars = 2 + 2 * kStages + 2 + 2 + 2;
  static constexpr int kSchedOffset = kBarOffset + kNumBars * 8 + 16;
  static constexpr int kSmemBytes = kSchedOffset + int(sizeof(TileSchedule)) + 1024;
};

template <typename T, int D, int VD, bool SPLIT, bool CL>
__global__ void __launch_bounds__(kBwdThreads, 2) bwd_dq_small_kernel(const __grid_constant__ BwdParams p) {
  using Cfg = DqSmallCfg<D, VD>;
  constexpr int kStages = Cfg::kStages;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  const uint32_t q_smem = smem_base;
  const uint32_t do_smem = smem_base + Cfg::kQBytes;
  const uint32_t ring = smem_base + Cfg::kRingOffset;
  const uint32_t bars = smem_base + Cfg::kBarOffset;
  const uint32_t bar_q_full = bars;
  const uint32_t bar_kv_full = bars + 16;
  const uint32_t bar_kv_empty = bar_kv_full + 8 * kStages;
  const uint32_t bar_s_full = bar_kv_empty + 8 * kStages;
  const uint32_t bar_p_ready = bar_s_full + 16;
  const uint32_t bar_final = bar_p_ready + 16;
  const uint32_t tmem_slot = bar_final + 16;
  volatile uint32_t* tmem_slot_gen =
      reinterpret_cast<volatile uint32_t*>(smem_gen + Cfg::kBarOffset + Cfg::kNumBars * 8);

  const int warp = threadIdx.x >> 5;
  const FaRule& rule = p.rule;
  const int b = int(blockIdx.x / p.n_blocks);                     // head-major: K/V stay in L2
  const BatchCoord bc = batch_coord<CL>(b, p.heads);
  const int pair = p.n_blocks - 1 - int(blockIdx.x % p.n_blocks);  // heavy (late) rows first
  const int q0 = pair * kBM;
  const int q_hi = min(q0 + kBM, p.nq) - 1;
  int kt_first, kt_last;
  fa_k_tile_range(rule, q0, q_hi, kBN, &kt_first, &kt_last);
  TileSchedule* sched = reinterpret_cast<TileSchedule*>(smem_gen + Cfg::kSchedOffset);
  {
    const int lo[1] = {q0};
    const int hi[1] = {q_hi};
    const bool valid[1] = {true};
    build_schedule(sched, rule, true, lo, hi, valid, 1, kt_first, kt_last, kBN, p.nk, kBwdThreads / 32);
  }

  if (warp == 8) {
    if (elect_one()) {
      prefetch_tensormap(&p.map_q);
      prefetch_tensormap(&p.map_k);
      prefetch_tensormap(&p.map_v);
      prefetch_tensormap(&p.map_do);
      prefetch_tensormap(&p.map_dq);
    }
  } else if (warp == 9) {
    if (elect_one()) {
      for (int i = 0; i < 2; ++i) {
        mbar_init(bar_q_full + 8 * i, 1);
        mbar_init(bar_s_full + 8 * i, 1);
        mbar_init(bar_p_ready + 8 * i, 2 * kBM);
        mbar_init(bar_final + 8 * i, 1);
      }
      for (int s = 0; s < kStages; ++s) {
        mbar_init(bar_kv_full + 8 * s, 1);
        mbar_init(bar_kv_empty + 8 * s, 1);
      }
      fence_barrier_init();
    }
  } else if (warp == 10) {
    tmem_alloc(tmem_slot, 256);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_gen;
  // TMEM columns (256 allocated -> two CTAs per SM): S [0, 64)  dP [64, 128)  dQ [128, +D); one 128-row Q tile,
  // both softmax warpgroups split the 64 key columns of every tile.
  // SPLIT (precise gradients): each warpgroup's 32 S columns hold dS as hi (first 16) + lo (next 16) fp16 pairs, its
  // first 16 dP columns hold P (fp16), and a second accumulator A2 = P K sits at [192, +D): the row sum D is
  // re-derived exactly as rowsum(P o dP) while the tiles stream by (the D handed in comes from the fp16-rounded O and is
  // off by up to ~5e-3, which P ~ 1 rows pass straight into dS), and dQ = scale (A1 - (D_exact - D) A2) at the end.
  static_assert(!SPLIT || 192 + D <= 256, "the P K accumulator of the precise variant needs 2 * D <= 128 columns");

  if (warp >= 8) {
    setmaxnreg_dec<32>();
    if (warp == 8) {
      if (elect_one()) {
        mbar_arrive_expect_tx(bar_q_full, Cfg::kQBytes + Cfg::kDoBytes);
        tile_load<CL>(q_smem, &p.map_q, bar_q_full, q0, kBM, D, bc);
        tile_load<CL>(do_smem, &p.map_do, bar_q_full, q0, kBM, VD, bc);
        int t = 0;
        TileIter it;
        it.init(sched, 1, kt_first, kt_last);
        int kt, tw, tb;
        while (it.next(&kt, &tw, &tb)) {
          const int s = t % kStages, u = t / kStages;
          mbar_wait(bar_kv_empty + 8 * s, (u & 1) ^ 1);
          mbar_arrive_expect_tx(bar_kv_full + 8 * s, Cfg::kStageBytes);
          tile_load<CL>(ring + s * Cfg::kStageBytes, &p.map_k, bar_kv_full + 8 * s, kt * kBN, kBN, D, bc);
          tile_load<CL>(ring + s * Cfg::kStageBytes + Cfg::kKBytes, &p.map_v, bar_kv_full + 8 * s, kt * kBN, kBN, VD, bc);
          ++t;
        }
      }
    } else if (warp == 9) {
      if (elect_one()) {
        TileIter it;
        it.init(sched, 1, kt_first, kt_last);
        const int n = it.count();
        constexpr uint32_t idesc_s = idesc_16<T>(kBM, kBN, tile_mn_major<CL>(true), tile_mn_major<CL>(true));
        constexpr uint32_t idesc_dq = idesc_16<T>(kBM, D, false, tile_mn_major<CL>(false));
        auto issue_s_dp = [&](int stage) {
          const uint32_t k_s = ring + stage * Cfg::kStageBytes, v_s = k_s + Cfg::kKBytes;
#pragma unroll
          for (int ks = 0; ks < D / 16; ++ks)
            mma_ss(tmem_base, tile_desc<CL>(q_smem, ks, kBM, D, true),
                   tile_desc<CL>(k_s, ks, kBN, D, true), idesc_s, ks > 0);
#pragma unroll
          for (int ks = 0; ks < VD / 16; ++ks)
            mma_ss(tmem_base + 64, tile_desc<CL>(do_smem, ks, kBM, VD, true),
                   tile_desc<CL>(v_s, ks, kBN, VD, true), idesc_s, ks > 0);
        };
        auto issue_dq = [&](int stage, bool accumulate) {
          const uint32_t k_s = ring + stage * Cfg::kStageBytes;
          // dS: warpgroup h wrote its 32 key columns as 16 packed columns at [32h, 32h+16)
#pragma unroll
          for (int ks = 0; ks < kBN / 16; ++ks)
            mma_ts(tmem_base + 128, tmem_base + (ks >> 1) * 32 + (ks & 1) * 8,
                   tile_desc<CL>(k_s, ks, kBN, D, false), idesc_dq, (accumulate || ks > 0) ? 1u : 0u);
          if constexpr (SPLIT) {   // the lo halves sit 16 columns behind their hi halves
#pragma unroll
            for (int ks = 0; ks < kBN / 16; ++ks)
              mma_ts(tmem_base + 128, tmem_base + (ks >> 1) * 32 + (ks & 1) * 8 + 16,
                     tile_desc<CL>(k_s, ks, kBN, D, false), idesc_dq, 1u);
#pragma unroll
            for (int ks = 0; ks < kBN / 16; ++ks)   // A2 += P K (P in the dP columns)
              mma_ts(tmem_base + 192, tmem_base + 64 + (ks >> 1) * 32 + (ks & 1) * 8,
                     tile_desc<CL>(k_s, ks, kBN, D, false), idesc_dq, (accumulate || ks > 0) ? 1u : 0u);
          }
        };
        if (n > 0) {
          mbar_wait(bar_kv_full + 0, 0);
          mbar_wait(bar_q_full, 0);
          tc_fence_after();
          issue_s_dp(0);
          mma_commit(bar_s_full);
          for (int j = 0; j < n; ++j) {
            const int sj = j % kStages, sn = (j + 1) % kStages;
            mbar_wait(bar_p_ready, j & 1);
            tc_fence_after();
            issue_dq(sj, j > 0);
            mma_commit(bar_kv_empty + 8 * sj);
            if (j + 1 < n) {
              mbar_wait(bar_kv_full + 8 * sn, ((j + 1) / kStages) & 1);
              tc_fence_after();
              issue_s_dp(sn);
              mma_commit(bar_s_full);
            } else {
              mma_commit(bar_final);
            }
          }
        }
      }
    }
  } else {
    setmaxnreg_inc<104>();
    const int x = warp >> 2;                 // key-column half in the main loop, channel half in the epilogue
    const int r = threadIdx.x & 127;         // query row
    const uint32_t lane_addr = uint32_t((warp & 3) * 32) << 16;
    const uint32_t t_s = tmem_base + lane_addr + x * 32;   // own 32 columns of S; dP at +64
    const uint32_t t_dq = tmem_base + lane_addr + 128;
    const int qi = q0 + r;
    const bool q_valid = qi < p.nq;
    const FaPos qpos = fa_pos(rule, rule.q, min(qi, p.nq - 1));
    const float lse2 = q_valid ? p.lse2[int64_t(b) * p.stat_pitch + qi] : __int_as_float(0x7f800000);
    const float dsum = q_valid ? p.dsum[int64_t(b) * p.stat_pitch + qi] : 0.f;
    const float scale_log2 = p.scale_log2;
    float d_exact = 0.f;   // SPLIT: this warpgroup's half of rowsum(P o dP)
    int j = 0;
    TileIter it;
    it.init(sched, 1, kt_first, kt_last);
    int kt, tw, tb;
    while (it.next(&kt, &tw, &tb)) {
      const int k0 = kt * kBN;
      const int k_hi = min(k0 + kBN, p.nk) - 1;
      const int cls = it.cls(0, tw, tb);
      const bool ragged = k0 + kBN > p.nk;
      mbar_wait(bar_s_full, j & 1);
      tc_fence_after();
      // masks first: nothing that may move registers between tcgen05.ld and tcgen05.wait::ld
      uint32_t okmask = 0xffffffffu;
      if (cls == FA_TILE_PARTIAL || ragged) {
        const int nvalid = k_hi - k0 + 1;
        if (rule.dims == 1 && rule.rule != 2) {
          int lo, hi;
          interval_1d(rule, true, qpos, k0, nvalid, &lo, &hi);
          okmask = interval_bits32(lo, hi, x * 32);
        } else {
          okmask = tile_mask32(rule, true, qpos, k0, x * 32, nvalid);
        }
      }
      float s[32], dp[32];
      tmem_ld32f(t_s, s);
      tmem_ld32f(t_s + 64, dp);
      tmem_wait_ld();
      uint32_t pk[16], pl[16], pp[16];
#pragma unroll
      for (int c = 0; c < 32; c += 2) {
        float p0 = ex2(fmaf(s[c], scale_log2, -lse2));
        float p1 = ex2(fmaf(s[c + 1], scale_log2, -lse2));
        p0 = (okmask >> c) & 1u ? p0 : 0.f;
        p1 = (okmask >> (c + 1)) & 1u ? p1 : 0.f;
        if constexpr (SPLIT) {
          d_exact = fmaf(p0, dp[c], d_exact);
          d_exact = fmaf(p1, dp[c + 1], d_exact);
          split2<T>(p0 * (dp[c] - dsum), p1 * (dp[c + 1] - dsum), pk[c >> 1], pl[c >> 1]);
          pp[c >> 1] = pack2<T>(p0, p1);
        } else {
          pk[c >> 1] = pack2<T>(p0 * (dp[c] - dsum), p1 * (dp[c + 1] - dsum));
        }
      }
      tmem_st16(t_s, pk);
      if constexpr (SPLIT) {
        tmem_st16(t_s + 16, pl);
        tmem_st16(t_s + 64, pp);
      }
      tmem_wait_st();
      tc_fence_before();
      mbar_arrive(bar_p_ready);
      ++j;
    }
    // epilogue: dQ = scale * acc -> fp16 -> smem [D][64] x2 -> TMA store; warpgroup x handles channels [32x, 32x+32)
    uint8_t* stage_gen = smem_gen;
    if (j > 0) {
      mbar_wait(bar_final, 0);
      tc_fence_after();
      float delta = 0.f;
      if constexpr (SPLIT) {
        // both halves of the exact row sum meet in shared memory (the dO tile is no longer read: every MMA has completed)
        float* dx = reinterpret_cast<float*>(smem_gen + Cfg::kQBytes);
        dx[x * kBM + r] = d_exact;
        named_bar_sync(2, 2 * kBM);
        const float d_full = dx[r] + dx[kBM + r];
        if (p.exact_d) {
          delta = d_full - dsum;
          if (x == 0 && q_valid) p.dsum_out[int64_t(b) * p.stat_pitch + qi] = d_full;
        }
      }
      for (int c = x; c < D / 32; c += 2) {
        float o[32];
        tmem_ld32f(t_dq + c * 32, o);
        tmem_wait_ld();
        if constexpr (SPLIT) {
          float o2[32];
          tmem_ld32f(t_dq + 64 + c * 32, o2);
          tmem_wait_ld();
#pragma unroll
          for (int e = 0; e < 32; ++e) o[e] = fmaf(-delta, o2[e], o[e]);
        }
        stage_row32<CL, T>(stage_gen, r, c * 32, kBM, D, o, p.scale);
      }
    } else {
      mbar_wait(bar_q_full, 0);
      for (int c = x * 32; c < D; c += 64) stage_row_zero<CL>(stage_gen, r, c, c + 32, kBM, D);
    }
    fence_proxy_async_smem();
    named_bar_sync(1, 2 * kBM);
    if (threadIdx.x == 0) {
      tile_store<CL>(&p.map_dq, q_smem, q0, kBM, D, p.nq, bc);
      tma_store_commit();
      tma_store_wait_read();
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 10) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 256);
  }
}


// =================================================================================================
// dK / dV kernel
// =================================================================================================
template <int D, int VD>
struct DkvCfg {
  static constexpr int kStages = 4;
  static constexpr int kKBytes = kBM * D * 2;     // resident K tile, also dK staging
  static constexpr int kVBytes = kBM * VD * 2;    // resident V tile, also dV staging
  static constexpr int kQBytes = kBN * D * 2;     // streamed Q sub-tile
  static constexpr int kDoBytes = kBN * VD * 2;
  static constexpr int kStatBytes = 2 * kBN * 4;  // LSE2[64] + D[64]
  static constexpr int kStageBytes = kQBytes + kDoBytes;
  static constexpr int kRingOffset = kKBytes + kVBytes;
  static constexpr int kStatOffset = kRingOffset + kStages * kStageBytes;
  static constexpr int kBarOffset = kStatOffset + kStages * kStatBytes;
  static constexpr int kNumBars = 1 + 2 * kStages + 2 + 2 + 1;
  static constexpr int kSchedOffset = kBarOffset + kNumBars * 8 + 16;
  static constexpr int kSmemBytes = kSchedOffset + int(sizeof(TileSchedule)) + 1024;
};

__device__ __forceinline__ void bulk_load_1d(uint32_t smem_dst, const void* gsrc, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_dst),
               "l"(reinterpret_cast<uint64_t>(gsrc)), "r"(bytes), "r"(bar)
               : "memory");
}

template <typename T, int D, int VD, bool SPLIT, bool CL>
__global__ void __launch_bounds__(kBwdThreads, 1) bwd_dkdv_kernel(const __grid_constant__ BwdParams p) {
  using Cfg = DkvCfg<D, VD>;
  constexpr int kStages = Cfg::kStages;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  const uint32_t k_smem = smem_base;
  const uint32_t v_smem = smem_base + Cfg::kKBytes;
  const uint32_t ring = smem_base + Cfg::kRingOffset;
  const uint32_t stat_smem = smem_base + Cfg::kStatOffset;
  const uint32_t bars = smem_base + Cfg::kBarOffset;
  const uint32_t bar_kv_res = bars;                          // resident K/V landed
  const uint32_t bar_full = bars + 8;                        // [kStages]
  const uint32_t bar_empty = bar_full + 8 * kStages;         // [kStages]
  const uint32_t bar_s_full = bar_empty + 8 * kStages;       // [2]
  const uint32_t bar_p_ready = bar_s_full + 16;              // [2]
  const uint32_t bar_final = bar_p_ready + 16;               // [1]
  const uint32_t tmem_slot = bar_final + 8;
  volatile uint32_t* tmem_slot_gen =
      reinterpret_cast<volatile uint32_t*>(smem_gen + Cfg::kBarOffset + Cfg::kNumBars * 8);
  const float* stat_gen = reinterpret_cast<const float*>(smem_gen + Cfg::kStatOffset);

  const int warp = threadIdx.x >> 5;
  const FaRule& rule = p.rule;
  const int b = int(blockIdx.x / p.n_blocks);     // head-major: Q/dO stay in L2
  const BatchCoord bc = batch_coord<CL>(b, p.heads);
  const int kblk = int(blockIdx.x % p.n_blocks);  // early key tiles are the heavy ones under causal
  const int k0 = kblk * kBM;
  const int k_hi = min(k0 + kBM, p.nk) - 1;
  int qt_first, qt_last;
  fa_q_tile_range(rule, k0, k_hi, kBN, &qt_first, &qt_last);
  TileSchedule* sched = reinterpret_cast<TileSchedule*>(smem_gen + Cfg::kSchedOffset);
  {
    const int lo[1] = {k0};
    const int hi[1] = {k_hi};
    const bool valid[1] = {true};
    build_schedule(sched, rule, false, lo, hi, valid, 1, qt_first, qt_last, kBN, p.nq, kBwdThreads / 32);
  }

  if (warp == 8) {
    if (elect_one()) {
      prefetch_tensormap(&p.map_q);
      prefetch_tensormap(&p.map_k);
      prefetch_tensormap(&p.map_v);
      prefetch_tensormap(&p.map_do);
      prefetch_tensormap(&p.map_dk);
      prefetch_tensormap(&p.map_dv);
    }
  } else if (warp == 9) {
    if (elect_one()) {
      mbar_init(bar_kv_res, 1);
      mbar_init(bar_final, 1);
      for (int i = 0; i < 2; ++i) {
        mbar_init(bar_s_full + 8 * i, 1);
        mbar_init(bar_p_ready + 8 * i, kBM);
      }
      for (int s = 0; s < kStages; ++s) {
        mbar_init(bar_full + 8 * s, 1);
        mbar_init(bar_empty + 8 * s, 1);
      }
      fence_barrier_init();
    }
  } else if (warp == 10) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_gen;
  // TMEM columns: S^T_x [x*64, +64)  dP^T_x [128+x*64, +64)  dV [256, +VD)  dK [384, +D)

  if (warp >= 8) {
    setmaxnreg_dec<56>();
    if (warp == 8) {
      if (elect_one()) {
        mbar_arrive_expect_tx(bar_kv_res, Cfg::kKBytes + Cfg::kVBytes);
        tile_load<CL>(k_smem, &p.map_k, bar_kv_res, k0, kBM, D, bc);
        tile_load<CL>(v_smem, &p.map_v, bar_kv_res, k0, kBM, VD, bc);
        int t = 0;
        TileIter it;
        it.init(sched, 1, qt_first, qt_last);
        int qt, tw, tb;
        while (it.next(&qt, &tw, &tb)) {
          const int s = t % kStages, u = t / kStages;
          mbar_wait(bar_empty + 8 * s, (u & 1) ^ 1);
          mbar_arrive_expect_tx(bar_full + 8 * s, Cfg::kStageBytes + Cfg::kStatBytes);
          tile_load<CL>(ring + s * Cfg::kStageBytes, &p.map_q, bar_full + 8 * s, qt * kBN, kBN, D, bc);
          tile_load<CL>(ring + s * Cfg::kStageBytes + Cfg::kQBytes, &p.map_do, bar_full + 8 * s, qt * kBN, kBN, VD, bc);
          const int64_t off = int64_t(b) * p.stat_pitch + qt * kBN;
          bulk_load_1d(stat_smem + s * Cfg::kStatBytes, p.lse2 + off, kBN * 4, bar_full + 8 * s);
          bulk_load_1d(stat_smem + s * Cfg::kStatBytes + kBN * 4, p.dsum + off, kBN * 4, bar_full + 8 * s);
          ++t;
        }
      }
    } else if (warp == 9) {
      if (elect_one()) {
        TileIter it;
        it.init(sched, 1, qt_first, qt_last);
        const int n = it.count();
        constexpr uint32_t idesc_st = idesc_16<T>(kBM, kBN, tile_mn_major<CL>(true), tile_mn_major<CL>(true));
        constexpr uint32_t idesc_dv = idesc_16<T>(kBM, VD, false, tile_mn_major<CL>(false));
        constexpr uint32_t idesc_dk = idesc_16<T>(kBM, D, false, tile_mn_major<CL>(false));
        auto issue_st_dpt = [&](int x, int stage) {
          const uint32_t q_s = ring + stage * Cfg::kStageBytes, do_s = q_s + Cfg::kQBytes;
#pragma unroll
          for (int ks = 0; ks < D / 16; ++ks)
            mma_ss(tmem_base + x * kBN, tile_desc<CL>(k_smem, ks, kBM, D, true),
                   tile_desc<CL>(q_s, ks, kBN, D, true), idesc_st, ks > 0);
#pragma unroll
          for (int ks = 0; ks < VD / 16; ++ks)
            mma_ss(tmem_base + 128 + x * kBN, tile_desc<CL>(v_smem, ks, kBM, VD, true),
                   tile_desc<CL>(do_s, ks, kBN, VD, true), idesc_st, ks > 0);
        };
        auto issue_dv_dk = [&](int x, int stage, bool accumulate) {
          const uint32_t q_s = ring + stage * Cfg::kStageBytes, do_s = q_s + Cfg::kQBytes;
#pragma unroll
          for (int ks = 0; ks < kBN / 16; ++ks)
            mma_ts(tmem_base + 256, tmem_base + x * kBN + ks * 8, tile_desc<CL>(do_s, ks, kBN, VD, false),
                   idesc_dv, (accumulate || ks > 0) ? 1u : 0u);
          if constexpr (SPLIT) {   // P^T lo halves: the 32 columns behind the packed hi halves
#pragma unroll
            for (int ks = 0; ks < kBN / 16; ++ks)
              mma_ts(tmem_base + 256, tmem_base + x * kBN + 32 + ks * 8, tile_desc<CL>(do_s, ks, kBN, VD, false),
                     idesc_dv, 1u);
          }
#pragma unroll
          for (int ks = 0; ks < kBN / 16; ++ks)
            mma_ts(tmem_base + 384, tmem_base + 128 + x * kBN + ks * 8, tile_desc<CL>(q_s, ks, kBN, D, false),
                   idesc_dk, (accumulate || ks > 0) ? 1u : 0u);
          if constexpr (SPLIT) {   // dS^T lo halves: the 32 columns behind the packed hi halves
#pragma unroll
            for (int ks = 0; ks < kBN / 16; ++ks)
              mma_ts(tmem_base + 384, tmem_base + 128 + x * kBN + 32 + ks * 8,
                     tile_desc<CL>(q_s, ks, kBN, D, false), idesc_dk, 1u);
          }
        };
        if (n > 0) {
          mbar_wait(bar_kv_res, 0);
          for (int t = 0; t < 2 && t < n; ++t) {
            mbar_wait(bar_full + 8 * (t % kStages), (t / kStages) & 1);
            tc_fence_after();
            issue_st_dpt(t & 1, t % kStages);
            mma_commit(bar_s_full + 8 * (t & 1));
          }
          for (int t = 0; t < n; ++t) {
            const int x = t & 1, st = t % kStages;
            mbar_wait(bar_p_ready + 8 * x, (t >> 1) & 1);
            tc_fence_after();
            issue_dv_dk(x, st, t > 0);
            mma_commit(bar_empty + 8 * st);
            if (t + 2 < n) {
              const int t2 = t + 2, s2 = t2 % kStages;
              mbar_wait(bar_full + 8 * s2, (t2 / kStages) & 1);
              tc_fence_after();
              issue_st_dpt(x, s2);
              mma_commit(bar_s_full + 8 * x);
            }
          }
          mma_commit(bar_final);
        }
      }
    }
  } else {
    setmaxnreg_inc<224>();
    const int x = warp >> 2;                 // ping-pong slot this warpgroup serves
    const int r = threadIdx.x & 127;         // key row
    const uint32_t lane_addr = uint32_t((warp & 3) * 32) << 16;
    const uint32_t t_s = tmem_base + lane_addr + x * kBN;
    const uint32_t t_dp = tmem_base + lane_addr + 128 + x * kBN;
    const int ki = k0 + r;
    const bool k_valid = ki < p.nk;
    const FaPos kpos = fa_pos(rule, rule.k, min(ki, p.nk - 1));
    const float scale_log2 = p.scale_log2;
    int t = 0;   // index over live sub-tiles (all), this WG handles those with (t & 1) == x
    TileIter it;
    it.init(sched, 1, qt_first, qt_last);
    int qt, tw, tb;
    while (it.next(&qt, &tw, &tb)) {
      if ((t & 1) != x) {
        ++t;
        continue;
      }
      const int st = t % kStages;
      const int q0 = qt * kBN;
      const int q_hi = min(q0 + kBN, p.nq) - 1;
      const int cls = it.cls(0, tw, tb);
      const bool ragged = (q0 + kBN > p.nq) || (k0 + kBM > p.nk);
      mbar_wait(bar_full + 8 * st, (t / kStages) & 1);   // stats visible to this thread
      mbar_wait(bar_s_full + 8 * x, (t >> 1) & 1);
      tc_fence_after();
      // masks first: nothing that may move registers between tcgen05.ld and tcgen05.wait::ld
      uint32_t okmask_lo = 0xffffffffu, okmask_hi = 0xffffffffu;
      if (cls == FA_TILE_PARTIAL || ragged) {
        okmask_lo = okmask_hi = 0u;
        if (k_valid) {
          const int nvalid = q_hi - q0 + 1;
          if (rule.dims == 1 && rule.rule != 2) {
            int lo, hi;
            interval_1d(rule, false, kpos, q0, nvalid, &lo, &hi);
            okmask_lo = interval_bits32(lo, hi, 0);
            okmask_hi = interval_bits32(lo, hi, 32);
          } else {
            okmask_lo = tile_mask32(rule, false, kpos, q0, 0, nvalid);
            okmask_hi = tile_mask32(rule, false, kpos, q0, 32, nvalid);
          }
        }
      }
      float s[64], dp[64];
      tmem_ld32f(t_s, &s[0]);
      tmem_ld32f(t_s + 32, &s[32]);
      tmem_ld32f(t_dp, &dp[0]);
      tmem_ld32f(t_dp + 32, &dp[32]);
      tmem_wait_ld();
      const float* lse_s = stat_gen + st * (2 * kBN);
      const float* dsum_s = lse_s + kBN;
      uint32_t pk[32], dk[32], dl[SPLIT ? 32 : 1], pl[SPLIT ? 32 : 1];
#pragma unroll
      for (int c = 0; c < 64; c += 2) {
        const uint32_t mword = c < 32 ? okmask_lo : okmask_hi;
        float p0 = ex2(fmaf(s[c], scale_log2, -lse_s[c]));
        float p1 = ex2(fmaf(s[c + 1], scale_log2, -lse_s[c + 1]));
        p0 = (mword >> (c & 31)) & 1u ? p0 : 0.f;
        p1 = (mword >> ((c + 1) & 31)) & 1u ? p1 : 0.f;
        if constexpr (SPLIT)
          split2<T>(p0, p1, pk[c >> 1], pl[c >> 1]);
        else
          pk[c >> 1] = pack2<T>(p0, p1);
        if constexpr (SPLIT)
          split2<T>(p0 * (dp[c] - dsum_s[c]), p1 * (dp[c + 1] - dsum_s[c + 1]), dk[c >> 1], dl[c >> 1]);
        else
          dk[c >> 1] = pack2<T>(p0 * (dp[c] - dsum_s[c]), p1 * (dp[c + 1] - dsum_s[c + 1]));
      }
      tmem_st32(t_s, pk);
      tmem_st32(t_dp, dk);
      if constexpr (SPLIT) {
        tmem_st32(t_s + 32, pl);
        tmem_st32(t_dp + 32, dl);
      }
      tmem_wait_st();
      tc_fence_before();
      mbar_arrive(bar_p_ready + 8 * x);
      ++t;
    }
    // how many live sub-tiles exist in total (t counted them all)
    // epilogue: warpgroup 0 stores dV, warpgroup 1 stores dK
    const int CH = x == 0 ? VD : D;
    const uint32_t t_acc = tmem_base + lane_addr + (x == 0 ? 256 : 384);
    const float out_scale = x == 0 ? 1.f : p.scale;
    uint8_t* stage_gen = smem_gen + (x == 0 ? Cfg::kKBytes : 0);
    if (t > 0) {
      mbar_wait(bar_final, 0);
      tc_fence_after();
      for (int c = 0; c < CH / 32; ++c) {
        float o[32];
        tmem_ld32f(t_acc + c * 32, o);
        tmem_wait_ld();
        stage_row32<CL, T>(stage_gen, r, c * 32, kBM, CH, o, out_scale);
      }
    } else {
      mbar_wait(bar_kv_res, 0);
      stage_row_zero<CL>(stage_gen, r, 0, CH, kBM, CH);
    }
    fence_proxy_async_smem();
    named_bar_sync(1 + x, kBM);
    if (r == 0) {
      if (x == 0)
        tile_store<CL>(&p.map_dv, v_smem, k0, kBM, VD, p.nk, bc);
      else
        tile_store<CL>(&p.map_dk, k_smem, k0, kBM, D, p.nk, bc);
      tma_store_commit();
      tma_store_wait_read();
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 10) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// =================================================================================================
// dK / dV kernel, small configuration (head_dim 64): one S^T / dP^T slot, both softmax warpgroups split
// the 64 query columns of every sub-tile, 256 TMEM columns and ~100 KB of shared memory -> two CTAs per SM
// =================================================================================================
template <int D, int VD>
struct DkvSmallCfg {
  static constexpr int kStages = 4;
  static constexpr int kKBytes = kBM * D * 2;     // resident K tile, also dK staging
  static constexpr int kVBytes = kBM * VD * 2;    // resident V tile, also dV staging
  static constexpr int kQBytes = kBN * D * 2;     // streamed Q sub-tile
  static constexpr int kDoBytes = kBN * VD * 2;
  static constexpr int kStatBytes = 2 * kBN * 4;  // LSE2[64] + D[64]
  static constexpr int kStageBytes = kQBytes + kDoBytes;
  static constexpr int kRingOffset = kKBytes + kVBytes;
  static constexpr int kStatOffset = kRingOffset + kStages * kStageBytes;
  static constexpr int kBarOffset = kStatOffset + kStages * kStatBytes;
  static constexpr int kNumBars = 1 + 2 * kStages + 2 + 2 + 1;
  static constexpr int kSchedOffset = kBarOffset + kNumBars * 8 + 16;
  static constexpr int kSmemBytes = kSchedOffset + int(sizeof(TileSchedule)) + 1024;
};

template <typename T, int D, int VD, bool SPLIT, bool CL>
__global__ void __launch_bounds__(kBwdThreads, 2) bwd_dkdv_small_kernel(const __grid_constant__ BwdParams p) {
  using Cfg = DkvSmallCfg<D, VD>;
  constexpr int kStages = Cfg::kStages;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  const uint32_t k_smem = smem_base;
  const uint32_t v_smem = smem_base + Cfg::kKBytes;
  const uint32_t ring = smem_base + Cfg::kRingOffset;
  const uint32_t stat_smem = smem_base + Cfg::kStatOffset;
  const uint32_t bars = smem_base + Cfg::kBarOffset;
  const uint32_t bar_kv_res = bars;                          // resident K/V landed
  const uint32_t bar_full = bars + 8;                        // [kStages]
  const uint32_t bar_empty = bar_full + 8 * kStages;         // [kStages]
  const uint32_t bar_s_full = bar_empty + 8 * kStages;       // [2] (only [0] used)
  const uint32_t bar_p_ready = bar_s_full + 16;              // [2]
  const uint32_t bar_final = bar_p_ready + 16;               // [1]
  const uint32_t tmem_slot = bar_final + 8;
  volatile uint32_t* tmem_slot_gen =
      reinterpret_cast<volatile uint32_t*>(smem_gen + Cfg::kBarOffset + Cfg::kNumBars * 8);
  const float* stat_gen = reinterpret_cast<const float*>(smem_gen + Cfg::kStatOffset);

  const int warp = threadIdx.x >> 5;
  const FaRule& rule = p.rule;
  const int b = int(blockIdx.x / p.n_blocks);     // head-major: Q/dO stay in L2
  const BatchCoord bc = batch_coord<CL>(b, p.heads);
  const int kblk = int(blockIdx.x % p.n_blocks);  // early key tiles are the heavy ones under causal
  const int k0 = kblk * kBM;
  const int k_hi = min(k0 + kBM, p.nk) - 1;
  int qt_first, qt_last;
  fa_q_tile_range(rule, k0, k_hi, kBN, &qt_first, &qt_last);
  TileSchedule* sched = reinterpret_cast<TileSchedule*>(smem_gen + Cfg::kSchedOffset);
  {
    const int lo[1] = {k0};
    const int hi[1] = {k_hi};
    const bool valid[1] = {true};
    build_schedule(sched, rule, false, lo, hi, valid, 1, qt_first, qt_last, kBN, p.nq, kBwdThreads / 32);
  }

  if (warp == 8) {
    if (elect_one()) {
      prefetch_tensormap(&p.map_q);
      prefetch_tensormap(&p.map_k);
      prefetch_tensormap(&p.map_v);
      prefetch_tensormap(&p.map_do);
      prefetch_tensormap(&p.map_dk);
      prefetch_tensormap(&p.map_dv);
    }
  } else if (warp == 9) {
    if (elect_one()) {
      mbar_init(bar_kv_res, 1);
      mbar_init(bar_final, 1);
      for (int i = 0; i < 2; ++i) {
        mbar_init(bar_s_full + 8 * i, 1);
        mbar_init(bar_p_ready + 8 * i, 2 * kBM);
      }
      for (int s = 0; s < kStages; ++s) {
        mbar_init(bar_full + 8 * s, 1);
        mbar_init(bar_empty + 8 * s, 1);
      }
      fence_barrier_init();
    }
  } else if (warp == 10) {
    tmem_alloc(tmem_slot, 256);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_gen;
  // TMEM columns (256 allocated, so that two CTAs share an SM): S^T [0, 64)  dP^T [64, 128)  dV [128, +VD)
  // dK [192, +D); one slot only: the second resident CTA provides the overlap that ping-pong slots give
  // the big configuration.

  if (warp >= 8) {
    setmaxnreg_dec<32>();
    if (warp == 8) {
      if (elect_one()) {
        mbar_arrive_expect_tx(bar_kv_res, Cfg::kKBytes + Cfg::kVBytes);
        tile_load<CL>(k_smem, &p.map_k, bar_kv_res, k0, kBM, D, bc);
        tile_load<CL>(v_smem, &p.map_v, bar_kv_res, k0, kBM, VD, bc);
        int t = 0;
        TileIter it;
        it.init(sched, 1, qt_first, qt_last);
        int qt, tw, tb;
        while (it.next(&qt, &tw, &tb)) {
          const int s = t % kStages, u = t / kStages;
          mbar_wait(bar_empty + 8 * s, (u & 1) ^ 1);
          mbar_arrive_expect_tx(bar_full + 8 * s, Cfg::kStageBytes + Cfg::kStatBytes);
          tile_load<CL>(ring + s * Cfg::kStageBytes, &p.map_q, bar_full + 8 * s, qt * kBN, kBN, D, bc);
          tile_load<CL>(ring + s * Cfg::kStageBytes + Cfg::kQBytes, &p.map_do, bar_full + 8 * s, qt * kBN, kBN, VD, bc);
          const int64_t off = int64_t(b) * p.stat_pitch + qt * kBN;
          bulk_load_1d(stat_smem + s * Cfg::kStatBytes, p.lse2 + off, kBN * 4, bar_full + 8 * s);
          bulk_load_1d(stat_smem + s * Cfg::kStatBytes + kBN * 4, p.dsum + off, kBN * 4, bar_full + 8 * s);
          ++t;
        }
      }
    } else if (warp == 9) {
      if (elect_one()) {
        TileIter it;
        it.init(sched, 1, qt_first, qt_last);
        const int n = it.count();
        constexpr uint32_t idesc_st = idesc_16<T>(kBM, kBN, tile_mn_major<CL>(true), tile_mn_major<CL>(true));
        constexpr uint32_t idesc_dv = idesc_16<T>(kBM, VD, false, tile_mn_major<CL>(false));
        constexpr uint32_t idesc_dk = idesc_16<T>(kBM, D, false, tile_mn_major<CL>(false));
        auto issue_st_dpt = [&](int stage) {
          const uint32_t q_s = ring + stage * Cfg::kStageBytes, do_s = q_s + Cfg::kQBytes;
#pragma unroll
          for (int ks = 0; ks < D / 16; ++ks)
            mma_ss(tmem_base, tile_desc<CL>(k_smem, ks, kBM, D, true),
                   tile_desc<CL>(q_s, ks, kBN, D, true), idesc_st, ks > 0);
#pragma unroll
          for (int ks = 0; ks < VD / 16; ++ks)
            mma_ss(tmem_base + 64, tile_desc<CL>(v_smem, ks, kBM, VD, true),
                   tile_desc<CL>(do_s, ks, kBN, VD, true), idesc_st, ks > 0);
        };
        auto issue_dv_dk = [&](int stage, bool accumulate) {
          const uint32_t q_s = ring + stage * Cfg::kStageBytes, do_s = q_s + Cfg::kQBytes;
          // P^T / dS^T: warpgroup h wrote its 32 query columns as 16 packed columns at [32h, 32h+16)
#pragma unroll
          for (int ks = 0; ks < kBN / 16; ++ks)
            mma_ts(tmem_base + 128, tmem_base + (ks >> 1) * 32 + (ks & 1) * 8,
                   tile_desc<CL>(do_s, ks, kBN, VD, false), idesc_dv, (accumulate || ks > 0) ? 1u : 0u);
          if constexpr (SPLIT) {   // P^T lo halves, 16 columns behind the hi halves
#pragma unroll
            for (int ks = 0; ks < kBN / 16; ++ks)
              mma_ts(tmem_base + 128, tmem_base + (ks >> 1) * 32 + (ks & 1) * 8 + 16,
                     tile_desc<CL>(do_s, ks, kBN, VD, false), idesc_dv, 1u);
          }
#pragma unroll
          for (int ks = 0; ks < kBN / 16; ++ks)
            mma_ts(tmem_base + 192, tmem_base + 64 + (ks >> 1) * 32 + (ks & 1) * 8,
                   tile_desc<CL>(q_s, ks, kBN, D, false), idesc_dk, (accumulate || ks > 0) ? 1u : 0u);
          if constexpr (SPLIT) {   // dS^T lo halves, 16 columns behind the hi halves
#pragma unroll
            for (int ks = 0; ks < kBN / 16; ++ks)
              mma_ts(tmem_base + 192, tmem_base + 64 + (ks >> 1) * 32 + (ks & 1) * 8 + 16,
                     tile_desc<CL>(q_s, ks, kBN, D, false), idesc_dk, 1u);
          }
        };
        if (n > 0) {
          mbar_wait(bar_kv_res, 0);
          mbar_wait(bar_full + 0, 0);
          tc_fence_after();
          issue_st_dpt(0);
          mma_commit(bar_s_full);
          for (int t = 0; t < n; ++t) {
            const int st = t % kStages;
            mbar_wait(bar_p_ready, t & 1);
            tc_fence_after();
            issue_dv_dk(st, t > 0);
            mma_commit(bar_empty + 8 * st);
            if (t + 1 < n) {
              const int t2 = t + 1, s2 = t2 % kStages;
              mbar_wait(bar_full + 8 * s2, (t2 / kStages) & 1);
              tc_fence_after();
              issue_st_dpt(s2);
              mma_commit(bar_s_full);
            }
          }
          mma_commit(bar_final);
        }
      }
    }
  } else {
    setmaxnreg_inc<104>();
    const int x = warp >> 2;                 // column half in the main loop, dV / dK role in the epilogue
    const int r = threadIdx.x & 127;         // key row
    const uint32_t lane_addr = uint32_t((warp & 3) * 32) << 16;
    const uint32_t t_s = tmem_base + lane_addr + x * 32;   // own 32 columns of S^T; dP^T at +64
    const int ki = k0 + r;
    const bool k_valid = ki < p.nk;
    const FaPos kpos = fa_pos(rule, rule.k, min(ki, p.nk - 1));
    const float scale_log2 = p.scale_log2;
    int t = 0;
    TileIter it;
    it.init(sched, 1, qt_first, qt_last);
    int qt, tw, tb;
    while (it.next(&qt, &tw, &tb)) {
      const int st = t % kStages;
      const int q0 = qt * kBN;
      const int q_hi = min(q0 + kBN, p.nq) - 1;
      const int cls = it.cls(0, tw, tb);
      const bool ragged = (q0 + kBN > p.nq) || (k0 + kBM > p.nk);
      mbar_wait(bar_full + 8 * st, (t / kStages) & 1);   // stats visible to this thread
      mbar_wait(bar_s_full, t & 1);
      tc_fence_after();
      // masks first: nothing that may move registers between tcgen05.ld and tcgen05.wait::ld
      uint32_t okmask = 0xffffffffu;
      if (cls == FA_TILE_PARTIAL || ragged) {
        okmask = 0u;
        if (k_valid) {
          const int nvalid = q_hi - q0 + 1;
          if (rule.dims == 1 && rule.rule != 2) {
            int lo, hi;
            interval_1d(rule, false, kpos, q0, nvalid, &lo, &hi);
            okmask = interval_bits32(lo, hi, x * 32);
          } else {
            okmask = tile_mask32(rule, false, kpos, q0, x * 32, nvalid);
          }
        }
      }
      float s[32], dp[32];
      tmem_ld32f(t_s, s);
      tmem_ld32f(t_s + 64, dp);
      tmem_wait_ld();
      const float4* lse4 = reinterpret_cast<const float4*>(stat_gen + st * (2 * kBN) + x * 32);
      const float4* dsum4 = lse4 + kBN / 4;
      uint32_t pk[16], dk[16], dl[16], pl[16];
#pragma unroll
      for (int c = 0; c < 32; c += 4) {
        const uint32_t mword = okmask >> c;
        const float4 ls = lse4[c >> 2];
        const float4 dd = dsum4[c >> 2];
        float p0 = ex2(fmaf(s[c], scale_log2, -ls.x));
        float p1 = ex2(fmaf(s[c + 1], scale_log2, -ls.y));
        float p2 = ex2(fmaf(s[c + 2], scale_log2, -ls.z));
        float p3 = ex2(fmaf(s[c + 3], scale_log2, -ls.w));
        p0 = mword & 1u ? p0 : 0.f;
        p1 = mword & 2u ? p1 : 0.f;
        p2 = mword & 4u ? p2 : 0.f;
        p3 = mword & 8u ? p3 : 0.f;
        if constexpr (SPLIT) {
          split2<T>(p0, p1, pk[c >> 1], pl[c >> 1]);
          split2<T>(p2, p3, pk[(c >> 1) + 1], pl[(c >> 1) + 1]);
        } else {
          pk[c >> 1] = pack2<T>(p0, p1);
          pk[(c >> 1) + 1] = pack2<T>(p2, p3);
        }
        if constexpr (SPLIT) {
          split2<T>(p0 * (dp[c] - dd.x), p1 * (dp[c + 1] - dd.y), dk[c >> 1], dl[c >> 1]);
          split2<T>(p2 * (dp[c + 2] - dd.z), p3 * (dp[c + 3] - dd.w), dk[(c >> 1) + 1], dl[(c >> 1) + 1]);
        } else {
          dk[c >> 1] = pack2<T>(p0 * (dp[c] - dd.x), p1 * (dp[c + 1] - dd.y));
          dk[(c >> 1) + 1] = pack2<T>(p2 * (dp[c + 2] - dd.z), p3 * (dp[c + 3] - dd.w));
        }
      }
      tmem_st16(t_s, pk);          // P^T  over the first 16 columns of this half of S^T
      tmem_st16(t_s + 64, dk);     // dS^T over the first 16 columns of this half of dP^T
      if constexpr (SPLIT) {
        tmem_st16(t_s + 16, pl);        // P^T lo halves
        tmem_st16(t_s + 64 + 16, dl);   // dS^T lo halves
      }
      tmem_wait_st();
      tc_fence_before();
      mbar_arrive(bar_p_ready);
      ++t;
    }
    // how many live sub-tiles exist in total (t counted them all)
    // epilogue: warpgroup 0 stores dV, warpgroup 1 stores dK
    const int CH = x == 0 ? VD : D;
    const uint32_t t_acc = tmem_base + lane_addr + (x == 0 ? 128 : 192);
    const float out_scale = x == 0 ? 1.f : p.scale;
    uint8_t* stage_gen = smem_gen + (x == 0 ? Cfg::kKBytes : 0);
    if (t > 0) {
      mbar_wait(bar_final, 0);
      tc_fence_after();
      for (int c = 0; c < CH / 32; ++c) {
        float o[32];
        tmem_ld32f(t_acc + c * 32, o);
        tmem_wait_ld();
        stage_row32<CL, T>(stage_gen, r, c * 32, kBM, CH, o, out_scale);
      }
    } else {
      mbar_wait(bar_kv_res, 0);
      stage_row_zero<CL>(stage_gen, r, 0, CH, kBM, CH);
    }
    fence_proxy_async_smem();
    named_bar_sync(1 + x, kBM);
    if (r == 0) {
      if (x == 0)
        tile_store<CL>(&p.map_dv, v_smem, k0, kBM, VD, p.nk, bc);
      else
        tile_store<CL>(&p.map_dk, k_smem, k0, kBM, D, p.nk, bc);
      tma_store_commit();
      tma_store_wait_read();
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 10) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 256);
  }
}


// LSE2 + D arrays (padded), rounded up so that the fp32 dQ scratch behind them is 256-byte aligned
static int64_t stat_pitch_of(int64_t nq) { return (nq + 3) & ~int64_t(3); }
static size_t stats_bytes(int64_t batch, int64_t nq) {
  return (size_t(2) * (batch * stat_pitch_of(nq) + kStatPad) * sizeof(float) + 255) & ~size_t(255);
}

static bool make_map_f32_sw128(CUtensorMap* map, const void* base, int64_t rows, int64_t cols, int box_cols,
                               int box_rows) {
  const uint64_t gdim[2] = {uint64_t(cols), uint64_t(rows)};
  const uint64_t gstride[1] = {uint64_t(cols) * 4};
  const uint32_t box[2] = {uint32_t(box_cols), uint32_t(box_rows)};
  return plan::tensor_map(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, base, gdim, gstride, box, CU_TENSOR_MAP_SWIZZLE_128B);
}

// =================================================================================================
// fused dQ / dK / dV kernel (D == 128)
// =================================================================================================
// Same CTA shape as bwd_dkdv_kernel (128 resident keys, 64-query sub-tiles in two ping-pong slots), but
// dQ is produced here as well, so S and dP are computed once instead of twice (5 GEMMs per tile pair
// instead of 7):
//     dQ^T[d, q] = K^T[d, keys] . dS^T[keys, q]
// A = the resident K tile re-read K-major, B = dS^T written by the softmax warps to shared memory in the
// MN-major 128B-swizzled layout (one 128-byte row of 64 queries per key), accumulator = the dP^T slot of
// the same ping-pong slot (the dP^T columns, free once the softmax warpgroup has read them). A fourth warpgroup drains the
// dQ^T accumulator and adds it into an fp32 [batch*D, nq] scratch tensor with TMA reduce-add
// (cp.reduce.async.bulk.tensor ... .add); bwd_dq_convert scales and rounds it to fp16 afterwards.
// (The order of the fp32 additions into the scratch tensor is not fixed, so dQ may differ in the last
// fp16 bit between runs; dK and dV are deterministic.)
#ifdef FA_DBG_TIMELINE
// developer-only (tools/timeline_bwd.py): clock64 stamps of CTA 0 -> g_dbg_bwd[role][t][event]
__device__ long long* g_dbg_bwd = nullptr;
#define FB_STAMP(role, j, ev)                                                                           \
  do {                                                                                                  \
    if (g_dbg_bwd && blockIdx.x == 0 && (j) < 128) g_dbg_bwd[((role) * 128 + (j)) * 4 + (ev)] = clock64(); \
  } while (0)
#else
#define FB_STAMP(role, j, ev)
#endif
constexpr int kFusedThreads = 512;

template <int D, int VD>
struct FusedCfg {
  static constexpr int kStages = 3;
  static constexpr int kKBytes = kBM * D * 2;
  static constexpr int kVBytes = kBM * VD * 2;
  static constexpr int kQBytes = kBN * D * 2;
  static constexpr int kDoBytes = kBN * VD * 2;
  static constexpr int kStatBytes = 2 * kBN * 4;
  static constexpr int kStageBytes = kQBytes + kDoBytes;
  static constexpr int kDsBytes = kBM * kBN * 2;       // dS^T tile, fp16, one per slot
  static constexpr int kRedBytes = D * 32 * 4;         // dQ^T staging: D rows x 32 queries fp32 (two of them)
  static constexpr int kRingOffset = kKBytes + kVBytes;
  static constexpr int kDsOffset = kRingOffset + kStages * kStageBytes;
  static constexpr int kRedOffset = kDsOffset + 2 * kDsBytes;
  static constexpr int kStatOffset = kRedOffset + 2 * kRedBytes;
  static constexpr int kBarOffset = kStatOffset + kStages * kStatBytes;
  static constexpr int kNumBars = 1 + 2 * kStages + 2 + 2 + 2 + 2 + 1;
  static constexpr int kSchedOffset = kBarOffset + kNumBars * 8 + 16;
  // no alignment slack: the dynamic shared window is declared 1024-byte aligned (checked at run time)
  static constexpr int kSmemBytes = kSchedOffset + int(sizeof(TileSchedule));
  static_assert(kSmemBytes <= 232448, "fused backward exceeds the 227 KB shared memory of an SM");
};

__device__ __forceinline__ void tma_reduce_add_2d(const void* map, uint32_t smem_src, int32_t x, int32_t y) {
  asm volatile("cp.reduce.async.bulk.tensor.2d.global.shared::cta.add.tile.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(map)),
               "r"(smem_src), "r"(x), "r"(y)
               : "memory");
}
__device__ __forceinline__ void bulk_wait_read_1() {
  asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
}
__device__ __forceinline__ void st_shared_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}

struct alignas(64) FusedParams {
  BwdParams base;
  CUtensorMap map_dq_acc;   // fp32 [batch*D, nq], box 32 x D, 128B swizzle
  // ACC (fa_backward_accumulate): dQ is ADDED into the caller's fp32 accumulator - the reduce-add above lands there
  // directly (scaled in the drain), so the scratch memset, the convert pass and the caller's fa_grad_accumulate pass
  // disappear. Problem pb adds into accumulator element pb % dq_fold (the K/V ring launches [Q_hi; Q_hi] pairs whose
  // two halves belong to the same accumulator). dK / dV are written as usual.
  int32_t dq_fold;
};

template <typename T, int D, int VD, bool CL, bool ACC>
__global__ void __launch_bounds__(kFusedThreads, 1) bwd_fused_kernel(const __grid_constant__ FusedParams fp) {
  using Cfg = FusedCfg<D, VD>;
  constexpr int kStages = Cfg::kStages;
  const BwdParams& p = fp.base;
  extern __shared__ __align__(1024) uint8_t smem_fused[];
  const uint32_t smem_base = smem_u32(smem_fused);
  if (smem_base & 1023u) __trap();   // swizzled tiles need 1024-byte alignment
  uint8_t* smem_gen = smem_fused;
  const uint32_t k_smem = smem_base;
  const uint32_t v_smem = smem_base + Cfg::kKBytes;
  const uint32_t ring = smem_base + Cfg::kRingOffset;
  const uint32_t ds_smem = smem_base + Cfg::kDsOffset;     // [2][kDsBytes]
  const uint32_t red_smem = smem_base + Cfg::kRedOffset;   // [2][kRedBytes]
  const uint32_t stat_smem = smem_base + Cfg::kStatOffset;
  const uint32_t bars = smem_base + Cfg::kBarOffset;
  const uint32_t bar_kv_res = bars;
  const uint32_t bar_full = bars + 8;                        // [kStages]
  const uint32_t bar_empty = bar_full + 8 * kStages;         // [kStages]
  const uint32_t bar_s_full = bar_empty + 8 * kStages;       // [2]
  const uint32_t bar_p_ready = bar_s_full + 16;              // [2]
  const uint32_t bar_dq_full = bar_p_ready + 16;             // [2]
  const uint32_t bar_dq_free = bar_dq_full + 16;             // [2]
  const uint32_t bar_final = bar_dq_free + 16;               // [1]
  const uint32_t tmem_slot = bar_final + 8;
  volatile uint32_t* tmem_slot_gen =
      reinterpret_cast<volatile uint32_t*>(smem_gen + Cfg::kBarOffset + Cfg::kNumBars * 8);
  const float* stat_gen = reinterpret_cast<const float*>(smem_gen + Cfg::kStatOffset);

  const int warp = threadIdx.x >> 5;
  const FaRule& rule = p.rule;
  const int b = int(blockIdx.x / p.n_blocks);
  const BatchCoord bc = batch_coord<CL>(b, p.heads);
  const int kblk = int(blockIdx.x % p.n_blocks);
  const int k0 = kblk * kBM;
  const int k_hi = min(k0 + kBM, p.nk) - 1;
  int qt_first, qt_last;
  fa_q_tile_range(rule, k0, k_hi, kBN, &qt_first, &qt_last);
  TileSchedule* sched = reinterpret_cast<TileSchedule*>(smem_gen + Cfg::kSchedOffset);
  {
    const int lo[1] = {k0};
    const int hi[1] = {k_hi};
    const bool valid[1] = {true};
    build_schedule(sched, rule, false, lo, hi, valid, 1, qt_first, qt_last, kBN, p.nq, kFusedThreads / 32);
  }

  if (warp == 8) {
    if (elect_one()) {
      prefetch_tensormap(&p.map_q);
      prefetch_tensormap(&p.map_k);
      prefetch_tensormap(&p.map_v);
      prefetch_tensormap(&p.map_do);
      prefetch_tensormap(&p.map_dk);
      prefetch_tensormap(&p.map_dv);
      prefetch_tensormap(&fp.map_dq_acc);
    }
  } else if (warp == 9) {
    if (elect_one()) {
      mbar_init(bar_kv_res, 1);
      mbar_init(bar_final, 1);
      for (int i = 0; i < 2; ++i) {
        mbar_init(bar_s_full + 8 * i, 1);
        mbar_init(bar_p_ready + 8 * i, 2 * kBM);
        mbar_init(bar_dq_full + 8 * i, 1);
        mbar_init(bar_dq_free + 8 * i, 128);
      }
      for (int s = 0; s < kStages; ++s) {
        mbar_init(bar_full + 8 * s, 1);
        mbar_init(bar_empty + 8 * s, 1);
      }
      fence_barrier_init();
    }
  } else if (warp == 10) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_gen;
  // TMEM columns: slot x: S^T_x [x*64, +64), later packed fp16 P^T_x [x*64, +32) and dS^T_x [x*64+32, +32);
  // dP^T_x [128+x*64, +64), later dQ^T_x (free once the softmax warpgroup has read dP^T);  dV [256, +VD);
  // dK [384, +D). S^T of the next sub-tile only has to wait for dV / dK of this one (in order on the
  // tensor pipe); dP^T of the next sub-tile waits for the dQ^T drain, one S^T product later.

  // register budget (512 threads x 128 at launch): softmax 8 warps x 184, drain 4 warps x 88, others 4 x 56
  if (warp >= 12) {
    setmaxnreg_dec<88>();
    // ---- dQ^T drain: TMEM -> registers -> swizzled staging tile -> TMA reduce-add into fp32 scratch
    const int rr = threadIdx.x - 384;   // channel row d
    const uint32_t lane_addr = uint32_t((warp & 3) * 32) << 16;
    int t = 0;
    TileIter it;
    it.init(sched, 1, qt_first, qt_last);
#ifdef FA_FUSED_NO_DQ
    it.init(sched, 1, 1, 0);
#endif
    int qt, tw, tb;
    while (it.next(&qt, &tw, &tb)) {
      const int x = t & 1;
      mbar_wait(bar_dq_full + 8 * x, (t >> 1) & 1);
      tc_fence_after();
      if (rr == 0) FB_STAMP(2, t, 0);
      // whole accumulator to registers first, so that the TMEM columns go back to the MMA warp at once
      uint32_t va[32], vb[32];
      tmem_ld32(tmem_base + lane_addr + 128 + x * kBN, va);
      tmem_ld32(tmem_base + lane_addr + 128 + x * kBN + 32, vb);
      tmem_wait_ld();
      tc_fence_before();
      mbar_arrive(bar_dq_free + 8 * x);
      if constexpr (ACC) {   // the accumulator holds finished gradients: the softmax scale goes in here
#pragma unroll
        for (int e = 0; e < 32; ++e) {
          va[e] = __float_as_uint(__uint_as_float(va[e]) * p.scale);
          vb[e] = __float_as_uint(__uint_as_float(vb[e]) * p.scale);
        }
      }
      if (rr == 0) FB_STAMP(2, t, 1);
      const uint32_t row_off = rr * 128;
      auto stage_half = [&](const uint32_t (&v)[32], int h) {
        const uint32_t stage = red_smem + h * Cfg::kRedBytes;
        if (rr == 0) bulk_wait_read_1();   // the reduce issued two groups ago has finished reading `stage`
        named_bar_sync(3, 128);
#pragma unroll
        for (int c = 0; c < 8; ++c)
          st_shared_v4(stage + row_off + ((c ^ (rr & 7)) << 4), v[4 * c], v[4 * c + 1], v[4 * c + 2], v[4 * c + 3]);
        fence_proxy_async_smem();
        named_bar_sync(3, 128);
        if (rr == 0) {
#ifndef FA_FUSED_NO_RED
          tma_reduce_add_2d(&fp.map_dq_acc, stage, qt * kBN + h * 32, (ACC ? b % fp.dq_fold : b) * D);
#endif
          tma_store_commit();
        }
      };
      stage_half(va, 0);
      stage_half(vb, 1);
      if (rr == 0) FB_STAMP(2, t, 2);
      ++t;
    }
    if (rr == 0) tma_store_wait_all();
  } else if (warp >= 8) {
    setmaxnreg_dec<56>();
    if (warp == 8) {
      if (elect_one()) {
        mbar_arrive_expect_tx(bar_kv_res, Cfg::kKBytes + Cfg::kVBytes);
        tile_load<CL>(k_smem, &p.map_k, bar_kv_res, k0, kBM, D, bc);
        tile_load<CL>(v_smem, &p.map_v, bar_kv_res, k0, kBM, VD, bc);
        int t = 0;
        TileIter it;
        it.init(sched, 1, qt_first, qt_last);
        int qt, tw, tb;
        while (it.next(&qt, &tw, &tb)) {
          const int s = t % kStages, u = t / kStages;
          mbar_wait(bar_empty + 8 * s, (u & 1) ^ 1);
          mbar_arrive_expect_tx(bar_full + 8 * s, Cfg::kStageBytes + Cfg::kStatBytes);
          tile_load<CL>(ring + s * Cfg::kStageBytes, &p.map_q, bar_full + 8 * s, qt * kBN, kBN, D, bc);
          tile_load<CL>(ring + s * Cfg::kStageBytes + Cfg::kQBytes, &p.map_do, bar_full + 8 * s, qt * kBN, kBN, VD, bc);
          const int64_t off = int64_t(b) * p.stat_pitch + qt * kBN;
          bulk_load_1d(stat_smem + s * Cfg::kStatBytes, p.lse2 + off, kBN * 4, bar_full + 8 * s);
          bulk_load_1d(stat_smem + s * Cfg::kStatBytes + kBN * 4, p.dsum + off, kBN * 4, bar_full + 8 * s);
          FB_STAMP(3, t, 3);
          ++t;
        }
      }
    } else if (warp == 9) {
      if (elect_one()) {
        TileIter it;
        it.init(sched, 1, qt_first, qt_last);
        const int n = it.count();
        constexpr uint32_t idesc_st = idesc_16<T>(kBM, kBN, tile_mn_major<CL>(true), tile_mn_major<CL>(true));
        constexpr uint32_t idesc_dv = idesc_16<T>(kBM, VD, false, tile_mn_major<CL>(false));
        constexpr uint32_t idesc_dk = idesc_16<T>(kBM, D, false, tile_mn_major<CL>(false));
        constexpr uint32_t idesc_dq = idesc_16<T>(D, kBN, tile_mn_major<CL>(false), true);
        auto issue_st = [&](int x, int stage) {
          const uint32_t q_s = ring + stage * Cfg::kStageBytes;
#pragma unroll
          for (int ks = 0; ks < D / 16; ++ks)
            mma_ss(tmem_base + x * kBN, tile_desc<CL>(k_smem, ks, kBM, D, true),
                   tile_desc<CL>(q_s, ks, kBN, D, true), idesc_st, ks > 0);
        };
        auto issue_dpt = [&](int x, int stage) {
          const uint32_t do_s = ring + stage * Cfg::kStageBytes + Cfg::kQBytes;
#pragma unroll
          for (int ks = 0; ks < VD / 16; ++ks)
            mma_ss(tmem_base + 128 + x * kBN, tile_desc<CL>(v_smem, ks, kBM, VD, true),
                   tile_desc<CL>(do_s, ks, kBN, VD, true), idesc_st, ks > 0);
        };
        auto issue_dq = [&](int x) {
#pragma unroll
          for (int ks = 0; ks < kBM / 16; ++ks)
            mma_ss(tmem_base + 128 + x * kBN,
                   tile_desc<CL>(k_smem, ks, kBM, D, false),
                   smem_desc_sw128(ds_smem + x * Cfg::kDsBytes + ks * 2048, 16, 1024), idesc_dq, ks > 0);
        };
        auto issue_dv_dk = [&](int x, int stage, bool accumulate) {
          const uint32_t q_s = ring + stage * Cfg::kStageBytes, do_s = q_s + Cfg::kQBytes;
#pragma unroll
          for (int ks = 0; ks < kBN / 16; ++ks)
            mma_ts(tmem_base + 256, tmem_base + x * kBN + (ks >> 1) * 32 + (ks & 1) * 8,
                   tile_desc<CL>(do_s, ks, kBN, VD, false), idesc_dv, (accumulate || ks > 0) ? 1u : 0u);
#pragma unroll
          for (int ks = 0; ks < kBN / 16; ++ks)
            mma_ts(tmem_base + 384, tmem_base + x * kBN + (ks >> 1) * 32 + 16 + (ks & 1) * 8,
                   tile_desc<CL>(q_s, ks, kBN, D, false), idesc_dk, (accumulate || ks > 0) ? 1u : 0u);
        };
        if (n > 0) {
          mbar_wait(bar_kv_res, 0);
          for (int t = 0; t < 2 && t < n; ++t) {
            mbar_wait(bar_full + 8 * (t % kStages), (t / kStages) & 1);
            tc_fence_after();
            issue_st(t & 1, t % kStages);
            issue_dpt(t & 1, t % kStages);
            mma_commit(bar_s_full + 8 * (t & 1));
          }
          for (int t = 0; t < n; ++t) {
            const int x = t & 1, st = t % kStages;
            mbar_wait(bar_p_ready + 8 * x, (t >> 1) & 1);
            tc_fence_after();
            FB_STAMP(1, t, 0);
#ifndef FA_FUSED_NO_DQ
            issue_dq(x);                       // first: its drain overlaps the dV / dK products
            mma_commit(bar_dq_full + 8 * x);
#endif
            FB_STAMP(3, t, 0);
            issue_dv_dk(x, st, t > 0);
            mma_commit(bar_empty + 8 * st);
            FB_STAMP(3, t, 1);
            if (t + 2 < n) {
              const int t2 = t + 2, s2 = t2 % kStages;
              mbar_wait(bar_full + 8 * s2, (t2 / kStages) & 1);
              tc_fence_after();
              FB_STAMP(3, t, 2);
              issue_st(x, s2);
              FB_STAMP(1, t, 1);
#ifndef FA_FUSED_NO_DQ
              mbar_wait(bar_dq_free + 8 * x, (t >> 1) & 1);   // dQ^T_x read out: dP^T_x may be overwritten
              tc_fence_after();
#endif
              FB_STAMP(1, t, 2);
              issue_dpt(x, s2);
              mma_commit(bar_s_full + 8 * x);
              FB_STAMP(1, t, 3);
            }
          }
          mma_commit(bar_final);
        }
      }
    }
  } else {
    setmaxnreg_inc<184>();
    // Both warpgroups work on EVERY sub-tile (no row reduction in the backward pass): warpgroup x takes the
    // query columns [32x, 32x+32) -> half the softmax latency on the S^T -> P^T/dS^T -> dV/dK/dQ chain.
    const int x = warp >> 2;                 // column half in the main loop; dV / dK role in the epilogue
    const int r = threadIdx.x & 127;         // key row
    const uint32_t lane_addr = uint32_t((warp & 3) * 32) << 16;
    const int ki = k0 + r;
    const bool k_valid = ki < p.nk;
    const FaPos kpos = fa_pos(rule, rule.k, min(ki, p.nk - 1));
    const float scale_log2 = p.scale_log2;
    int t = 0;
    TileIter it;
    it.init(sched, 1, qt_first, qt_last);
    int qt, tw, tb;
    while (it.next(&qt, &tw, &tb)) {
      const int slot = t & 1;
      const int st = t % kStages;
      const int q0 = qt * kBN;
      const int q_hi = min(q0 + kBN, p.nq) - 1;
      const int cls = it.cls(0, tw, tb);
      const bool ragged = (q0 + kBN > p.nq) || (k0 + kBM > p.nk);
      const uint32_t t_s = tmem_base + lane_addr + slot * kBN + x * 32;   // own 32 columns of S^T (dP^T at +128)
      mbar_wait(bar_full + 8 * st, (t / kStages) & 1);   // stats visible to this thread
      mbar_wait(bar_s_full + 8 * slot, (t >> 1) & 1);
      tc_fence_after();
      if (r == 0) FB_STAMP(0, t, 0);
      // masks first: nothing that may move registers between tcgen05.ld and tcgen05.wait::ld
      uint32_t okmask = 0xffffffffu;
      if (cls == FA_TILE_PARTIAL || ragged) {
        okmask = 0u;
        if (k_valid) {
          const int nvalid = q_hi - q0 + 1;
          if (rule.dims == 1 && rule.rule != 2) {
            int lo, hi;
            interval_1d(rule, false, kpos, q0, nvalid, &lo, &hi);
            okmask = interval_bits32(lo, hi, x * 32);
          } else {
            okmask = tile_mask32(rule, false, kpos, q0, x * 32, nvalid);
          }
        }
      }
      float s[32], dp[32];
      tmem_ld32f(t_s, s);
      tmem_ld32f(t_s + 128, dp);
      tmem_wait_ld();
      if (r == 0) FB_STAMP(0, t, 1);
      const float4* lse4 = reinterpret_cast<const float4*>(stat_gen + st * (2 * kBN) + x * 32);
      const float4* dsum4 = lse4 + kBN / 4;
      uint32_t pk[16], dk[16];
      if (okmask == 0xffffffffu) {
#pragma unroll
        for (int c = 0; c < 32; c += 4) {
          const float4 ls = lse4[c >> 2];
          const float4 dd = dsum4[c >> 2];
          const float p0 = ex2(fmaf(s[c], scale_log2, -ls.x));
          const float p1 = ex2(fmaf(s[c + 1], scale_log2, -ls.y));
          const float p2 = ex2(fmaf(s[c + 2], scale_log2, -ls.z));
          const float p3 = ex2(fmaf(s[c + 3], scale_log2, -ls.w));
          pk[c >> 1] = pack2<T>(p0, p1);
          pk[(c >> 1) + 1] = pack2<T>(p2, p3);
          dk[c >> 1] = pack2<T>(p0 * (dp[c] - dd.x), p1 * (dp[c + 1] - dd.y));
          dk[(c >> 1) + 1] = pack2<T>(p2 * (dp[c + 2] - dd.z), p3 * (dp[c + 3] - dd.w));
        }
      } else {
#pragma unroll
        for (int c = 0; c < 32; c += 4) {
          const uint32_t mword = okmask >> c;
          const float4 ls = lse4[c >> 2];
          const float4 dd = dsum4[c >> 2];
          float p0 = ex2(fmaf(s[c], scale_log2, -ls.x));
          float p1 = ex2(fmaf(s[c + 1], scale_log2, -ls.y));
          float p2 = ex2(fmaf(s[c + 2], scale_log2, -ls.z));
          float p3 = ex2(fmaf(s[c + 3], scale_log2, -ls.w));
          p0 = mword & 1u ? p0 : 0.f;
          p1 = mword & 2u ? p1 : 0.f;
          p2 = mword & 4u ? p2 : 0.f;
          p3 = mword & 8u ? p3 : 0.f;
          pk[c >> 1] = pack2<T>(p0, p1);
          pk[(c >> 1) + 1] = pack2<T>(p2, p3);
          dk[c >> 1] = pack2<T>(p0 * (dp[c] - dd.x), p1 * (dp[c + 1] - dd.y));
          dk[(c >> 1) + 1] = pack2<T>(p2 * (dp[c + 2] - dd.z), p3 * (dp[c + 3] - dd.w));
        }
      }
      if (r == 0) FB_STAMP(0, t, 2);
      tmem_st16(t_s, pk);           // P^T (fp16 pairs) over the first 16 of this half's S^T columns
      tmem_st16(t_s + 16, dk);      // dS^T over the other 16
      const uint32_t ds_row = ds_smem + slot * Cfg::kDsBytes + r * 128;
#pragma unroll
      for (int c = 0; c < 4; ++c)
        st_shared_v4(ds_row + (((x * 4 + c) ^ (r & 7)) << 4), dk[4 * c], dk[4 * c + 1], dk[4 * c + 2], dk[4 * c + 3]);
      fence_proxy_async_smem();
      tmem_wait_st();
      tc_fence_before();
      mbar_arrive(bar_p_ready + 8 * slot);
      if (r == 0) FB_STAMP(0, t, 3);
      ++t;
    }
    // epilogue: warpgroup 0 stores dV, warpgroup 1 stores dK (staged over the resident V / K tiles)
    const int CH = x == 0 ? VD : D;
    const uint32_t t_acc = tmem_base + lane_addr + (x == 0 ? 256 : 384);
    const float out_scale = x == 0 ? 1.f : p.scale;
    {
      uint8_t* stage_gen = smem_gen + (x == 0 ? Cfg::kKBytes : 0);
      if (t > 0) {
        mbar_wait(bar_final, 0);
        tc_fence_after();
        for (int c = 0; c < CH / 32; ++c) {
          float o[32];
          tmem_ld32f(t_acc + c * 32, o);
          tmem_wait_ld();
          stage_row32<CL, T>(stage_gen, r, c * 32, kBM, CH, o, out_scale);
        }
      } else {
        mbar_wait(bar_kv_res, 0);
        stage_row_zero<CL>(stage_gen, r, 0, CH, kBM, CH);
      }
      fence_proxy_async_smem();
      named_bar_sync(1 + x, kBM);
      if (r == 0) {
        if (x == 0)
          tile_store<CL>(&p.map_dv, v_smem, k0, kBM, VD, p.nk, bc);
        else
          tile_store<CL>(&p.map_dk, k_smem, k0, kBM, D, p.nk, bc);
        tma_store_commit();
        tma_store_wait_read();
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 10) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// dQ = T(scale * dQ_acc); 8 elements per thread
template <typename T>
__global__ void bwd_dq_convert(const float4* __restrict__ acc, uint4* __restrict__ dq, int64_t n8, float scale) {
  for (int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; i < n8; i += int64_t(gridDim.x) * blockDim.x) {
    const float4 a = acc[2 * i], c = acc[2 * i + 1];
    uint4 o;
    o.x = pack2<T>(a.x * scale, a.y * scale);
    o.y = pack2<T>(a.z * scale, a.w * scale);
    o.z = pack2<T>(c.x * scale, c.y * scale);
    o.w = pack2<T>(c.z * scale, c.w * scale);
    dq[i] = o;
  }
}

// channel-last dQ: the fused kernel's scratch stays [batch * 128][pitch] fp32 (its drain is layout-independent); this
// pass scales, rounds and transposes 64 positions x 128 channels per block through shared memory into
// [outer][q][heads][128] T
template <typename T>
__global__ void __launch_bounds__(256) bwd_dq_convert_cl(const float* __restrict__ acc, T* __restrict__ dq,
                                                         int64_t batch, int32_t nq, int64_t pitch, int32_t heads,
                                                         float scale) {
  constexpr int kPitch = 130;   // halves per staged position row: 4-byte aligned rows, 2-way bank conflicts at most
  __shared__ T tile[64 * kPitch];
  const int q0 = blockIdx.x * 64;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int q = q0 + 2 * lane;
  for (int64_t b = blockIdx.y; b < batch; b += gridDim.y) {   // gridDim.y is capped at 65535
    for (int d = warp; d < 128; d += 8) {
      float2 v = make_float2(0.f, 0.f);
      if (q < pitch) v = *reinterpret_cast<const float2*>(acc + (b * 128 + d) * pitch + q);   // pitch is even
      tile[(2 * lane) * kPitch + d] = from_acc<T>(v.x * scale);
      tile[(2 * lane + 1) * kPitch + d] = from_acc<T>(v.y * scale);
    }
    __syncthreads();
    const int64_t ob = b / heads, h = b % heads;
    for (int r = warp; r < 64 && q0 + r < nq; r += 8) {
      Pair<T>* dst = reinterpret_cast<Pair<T>*>(dq + ((ob * nq + q0 + r) * heads + h) * 128);
      const Pair<T>* src = reinterpret_cast<const Pair<T>*>(tile + r * kPitch);
      dst[lane] = src[lane];
      dst[lane + 32] = src[lane + 32];
    }
    __syncthreads();   // the tile is reused by the next batch element
  }
}

// fa_set_grad_precision(0): which problems get the split-operand ("precise") backward on their own. The operand rounding
// (and the D = rowsum(dO o O) taken from the fp16-rounded O) only matters where P is large, i.e. where rows attend few
// keys and a key collects many such rows; measured without it: 4.2e-3 on dK at 1000 queries x 88 keys (causal,
// scale_end), 2.1e-3 on 2-D strided windows of 2..3 positions, 2.005e-3 at 2135 heads x 64 x 64 causal. The precise
// kernels cost ~12 % on the HBM-bound workloads (S1, S2, C3: profiles/r2_grad_precision.md), so problems whose rows are
// long (P small) keep the plain ones.
static bool precise_auto(const FaRule& r) {
  const int64_t nq = r.q.total, nk = r.k.total;
  int64_t row_max = nk;   // upper bound on the keys one row attends
  if (r.rule == 2) {
    const int64_t ext[2] = {r.ref0, r.ref1};
    int64_t win = 1;
    for (int i = 0; i < r.dims; ++i) {
      const int64_t per_dim = std::min<int64_t>(2 * int64_t(r.window) - 1, 2 * ((ext[i] - 1) >> r.log2_stride) + 1);
      win = std::min<int64_t>(win * per_dim, nk);
    }
    row_max = win;
  }
  if (row_max <= 32) return true;                       // every row is short: P ~ 1/16 and larger everywhere
  const bool causal_type = r.rule == 1 || (r.rule == 2 && r.causal);
  // causal rules: the first rows of every key attend one, two, ... keys; one such row per key is harmless (measured
  // 1.2e-3 at the C2 shape), nq / nk of them per key are not, and in short sequences they are all there is
  return causal_type && (nk <= 128 || nq >= 4 * nk);
}

// ---- host side ---------------------------------------------------------------------------------
// Tensor maps of one kernel. Channel-first boxes are 64 positions x the kernel's channels for every kernel; a
// channel-last box is 64 channels x the tile's rows, which differ per kernel: rq rows for the q-length tensors
// (Q, dO, dQ), rk for the k-length ones.
template <typename T, int D, int VD, bool CL>
static bool bwd_maps(BwdParams* p, const LaunchArgs& a, int rq, int rk) {
  const int nq = a.rule.q.total, nk = a.rule.k.total;
  constexpr CUtensorMapDataType dt = Elt16<T>::kTmaType;
  if constexpr (CL) {
    const int64_t heads = a.heads, outer = a.batch / heads;
    return make_map_cl(&p->map_q, a.q, outer, heads, a.d, nq, rq, dt) && make_map_cl(&p->map_k, a.k, outer, heads, a.d, nk, rk, dt) &&
           make_map_cl(&p->map_v, a.v, outer, heads, a.v_d, nk, rk, dt) &&
           make_map_cl(&p->map_do, a.d_o, outer, heads, a.v_d, nq, rq, dt) &&
           make_map_cl(&p->map_dq, a.d_q, outer, heads, a.d, nq, rq, dt) &&
           make_map_cl(&p->map_dk, a.d_k, outer, heads, a.d, nk, rk, dt) &&
           make_map_cl(&p->map_dv, a.d_v, outer, heads, a.v_d, nk, rk, dt);
  } else {
    const int64_t qp = a.q_pitch ? a.q_pitch : nq, kp = a.k_pitch ? a.k_pitch : nk;
    return make_map_3d(&p->map_q, a.q, a.batch, a.d, nq, qp, D, true, dt) &&
           make_map_3d(&p->map_k, a.k, a.batch, a.d, nk, kp, D, true, dt) &&
           make_map_3d(&p->map_v, a.v, a.batch, a.v_d, nk, kp, VD, true, dt) &&
           make_map_3d(&p->map_do, a.d_o, a.batch, a.v_d, nq, qp, VD, true, dt) &&
           make_map_3d(&p->map_dq, a.d_q, a.batch, a.d, nq, qp, D, false, dt) &&
           make_map_3d(&p->map_dk, a.d_k, a.batch, a.d, nk, kp, D, false, dt) &&
           make_map_3d(&p->map_dv, a.d_v, a.batch, a.v_d, nk, kp, VD, false, dt);
  }
}

// D, VD: the kernels' padded channel counts (a.d <= D, a.v_d <= VD; the tensor maps zero-fill / clip the rest)
template <typename T, int D, int VD, bool CL>
cudaError_t launch_bwd(const LaunchArgs& a, cudaStream_t stream) {
  constexpr bool kBf16 = std::is_same<T, __nv_bfloat16>::value;
  BwdParams p;
  const int nq = a.rule.q.total, nk = a.rule.k.total;
  // row pitch of the fused kernel's fp32 dQ scratch (and, channel-first, of the dQ tensor the convert pass writes)
  const int64_t qp = CL ? ((int64_t(nq) + 7) & ~int64_t(7)) : (a.q_pitch ? a.q_pitch : nq);
  // fa_set_grad_precision: 1 = dS as hi + lo fp16 pairs everywhere (head_dim 128 then runs the two-kernel backward),
  // 2 = never, 0 = automatic: on for every path but the fused head_dim-128 kernel, whose TMEM has no room for the lo
  // halves and whose shapes (long rows, small P) measure inside the 2e-3 bar without them
  const bool fused_shape = D == 128 && a.d == 128;
  const bool split = a.grad_split == 1 || (a.grad_split == 0 && !fused_shape && precise_auto(a.rule));
  float* lse2 = reinterpret_cast<float*>(a.workspace);
  const int64_t sp = stat_pitch_of(nq);
  float* dsum = lse2 + (a.batch * sp + kStatPad);
  p.rule = a.rule;
  p.lse2 = lse2;
  p.dsum = dsum;
  p.nq = nq;
  p.nk = nk;
  p.batch = int32_t(a.batch);
  p.heads = CL ? a.heads : 1;
  p.stat_pitch = int32_t(sp);
  // the exact row sum needs every key of a row in this call (a ring block sees a key shard only)
  p.exact_d = (split && !a.partial_keys) ? 1 : 0;
  p.dsum_out = dsum;
  p.scale = 1.f / sqrtf(float(a.d));
  p.scale_log2 = p.scale * kLog2eB;
  {
    // statistics from the caller's own (dense) O and dO
    const int64_t total = a.batch * sp;
    ScopedKernel timed(CL ? (kBf16 ? "bwd_prep_bf16_cl" : "bwd_prep_f16_cl") : (kBf16 ? "bwd_prep_bf16" : "bwd_prep_f16"), stream);
    if constexpr (CL) {
      const int64_t outer = a.batch / a.heads;
      const int chunks = a.v_d / 8;
      const int64_t rows = outer * nq * int64_t(a.heads);
      auto go = [&](auto kern, int G) {
        const int blocks = int(std::min<int64_t>((rows * G + 255) / 256, 148 * 16));
        kern<<<std::max(blocks, 1), 256, 0, stream>>>((const T*)a.o, (const T*)a.prep_d_o, (const float*)a.l,
                                                     (const T*)a.m, lse2, dsum, outer, a.heads, a.v_d, nq, int32_t(sp));
      };
      if (chunks <= 1) go(bwd_prep_f16_cl<T, 1>, 1);
      else if (chunks <= 2) go(bwd_prep_f16_cl<T, 2>, 2);
      else if (chunks <= 4) go(bwd_prep_f16_cl<T, 4>, 4);
      else if (chunks <= 8) go(bwd_prep_f16_cl<T, 8>, 8);
      else go(bwd_prep_f16_cl<T, 16>, 16);
    } else if (nq % 2 == 0 && (reinterpret_cast<uintptr_t>(a.o) & 3) == 0 &&
               (reinterpret_cast<uintptr_t>(a.prep_d_o) & 3) == 0) {
      const int blocks = int(std::min<int64_t>((total / 2 + 255) / 256, 148 * 16));
      bwd_prep_f16<T><<<blocks, 256, 0, stream>>>((const T*)a.o, (const T*)a.prep_d_o, (const float*)a.l,
                                               (const T*)a.m, lse2, dsum, a.batch, a.v_d, nq, int32_t(sp));
    } else {
      const int blocks = int(std::min<int64_t>((total + 255) / 256, 148 * 16));
      bwd_prep_f16_any<T><<<blocks, 256, 0, stream>>>((const T*)a.o, (const T*)a.prep_d_o, (const float*)a.l,
                                                   (const T*)a.m, lse2, dsum, a.batch, a.v_d, nq, int32_t(sp));
    }
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
  }
  if constexpr (D == 128) {
    if (a.variant != 4 && !split && fused_shape) {
      // fused dQ/dK/dV: fp32 dQ scratch behind the row statistics, with the row pitch of the dQ tensor the convert pass
      // writes (the padded pitch when the q side is packed; the columns past nq only ever receive zeros)
      if (!bwd_maps<T, D, VD, CL>(&p, a, kBN, kBM)) return cudaErrorInvalidValue;
      if constexpr (!CL) {
        if (a.grad_acc) {
          // dQ added into the caller's fp32 accumulator through the kernel's own reduce-add: no scratch, no memset, no
          // convert pass (dK / dV: fp16 tensors as usual)
          FusedParams fp;
          fp.base = p;
          fp.dq_fold = int32_t(a.dq_fold);
          if (!make_map_f32_sw128(&fp.map_dq_acc, a.d_q, a.dq_fold * D, nq, 32, D)) return cudaErrorInvalidValue;
          auto kern = bwd_fused_kernel<T, D, VD, false, true>;
          cudaError_t e = plan::ensure_smem(kern, FusedCfg<D, VD>::kSmemBytes);
          if (e != cudaSuccess) return e;
          fp.base.n_blocks = (nk + kBM - 1) / kBM;
          ScopedKernel timed((kBf16 ? "bwd_fused_bf16_sm100_acc" : "bwd_fused_f16_sm100_acc"), stream);
          kern<<<unsigned(int64_t(fp.base.n_blocks) * p.batch), kFusedThreads, FusedCfg<D, VD>::kSmemBytes, stream>>>(fp);
          return cudaGetLastError();
        }
      }
      float* acc = reinterpret_cast<float*>(reinterpret_cast<char*>(a.workspace) + bwd_layout(a).off_acc);
      const size_t acc_bytes = size_t(a.batch) * D * qp * sizeof(float);
      FusedParams fp;
      fp.base = p;
      fp.dq_fold = 1;
      if (!make_map_f32_sw128(&fp.map_dq_acc, acc, a.batch * D, qp, 32, D)) return cudaErrorInvalidValue;
      {
        ScopedKernel timed("bwd_dq_zero", stream);
        cudaError_t e = cudaMemsetAsync(acc, 0, acc_bytes, stream);
        if (e != cudaSuccess) return e;
      }
      {
        auto kern = bwd_fused_kernel<T, D, VD, CL, false>;
        cudaError_t e =
            plan::ensure_smem(kern, FusedCfg<D, VD>::kSmemBytes);
        if (e != cudaSuccess) return e;
        fp.base.n_blocks = (nk + kBM - 1) / kBM;
        ScopedKernel timed(CL ? (kBf16 ? "bwd_fused_bf16_sm100_cl" : "bwd_fused_f16_sm100_cl") : (kBf16 ? "bwd_fused_bf16_sm100" : "bwd_fused_f16_sm100"), stream);
        kern<<<unsigned(int64_t(fp.base.n_blocks) * p.batch), kFusedThreads, FusedCfg<D, VD>::kSmemBytes, stream>>>(fp);
        e = cudaGetLastError();
        if (e != cudaSuccess) return e;
      }
      if constexpr (CL) {
        ScopedKernel timed((kBf16 ? "bwd_dq_convert_bf16_cl" : "bwd_dq_convert_cl"), stream);
        bwd_dq_convert_cl<T><<<dim3(unsigned((nq + 63) / 64), unsigned(std::min<int64_t>(a.batch, 65535))), 256, 0, stream>>>(
            acc, reinterpret_cast<T*>(a.d_q), a.batch, nq, qp, a.heads, p.scale);
        return cudaGetLastError();
      } else {
        const int64_t n8 = a.batch * int64_t(D) * qp / 8;
        const int blocks = int(std::min<int64_t>((n8 + 255) / 256, 148 * 16));
        ScopedKernel timed((kBf16 ? "bwd_dq_convert_bf16" : "bwd_dq_convert"), stream);
        bwd_dq_convert<T><<<blocks, 256, 0, stream>>>(reinterpret_cast<const float4*>(acc),
                                                   reinterpret_cast<uint4*>(a.d_q), n8, p.scale);
        return cudaGetLastError();
      }
    }
  }
  if (a.grad_acc) return cudaErrorNotSupported;   // only the fused kernel accumulates (checked by the caller)
  if (!bwd_maps<T, D, VD, CL>(&p, a, kBM, kBN)) return cudaErrorInvalidValue;   // dQ kernels: resident queries
  bool dq_done = false;
  if constexpr (D == 64 && VD == 64) {
    if (a.variant != 4) {
      auto kern = split ? bwd_dq_small_kernel<T, D, VD, true, CL> : bwd_dq_small_kernel<T, D, VD, false, CL>;
      cudaError_t e =
          plan::ensure_smem(kern, DqSmallCfg<D, VD>::kSmemBytes);
      if (e != cudaSuccess) return e;
      p.n_blocks = (nq + kBM - 1) / kBM;
      ScopedKernel timed(CL ? (kBf16 ? "bwd_dq_bf16_sm100_2cta_cl" : "bwd_dq_f16_sm100_2cta_cl") : (kBf16 ? "bwd_dq_bf16_sm100_2cta" : "bwd_dq_f16_sm100_2cta"), stream);
      kern<<<unsigned(int64_t(p.n_blocks) * p.batch), kBwdThreads, DqSmallCfg<D, VD>::kSmemBytes, stream>>>(p);
      e = cudaGetLastError();
      if (e != cudaSuccess) return e;
      dq_done = true;
    }
  }
  if (!dq_done) {
    auto kern = split ? bwd_dq_kernel<T, D, VD, true, CL> : bwd_dq_kernel<T, D, VD, false, CL>;
    cudaError_t e = plan::ensure_smem(kern, DqCfg<D, VD>::kSmemBytes);
    if (e != cudaSuccess) return e;
    p.n_blocks = (nq + 2 * kBM - 1) / (2 * kBM);
    ScopedKernel timed(CL ? (kBf16 ? "bwd_dq_bf16_sm100_cl" : "bwd_dq_f16_sm100_cl") : (kBf16 ? "bwd_dq_bf16_sm100" : "bwd_dq_f16_sm100"), stream);
    kern<<<unsigned(int64_t(p.n_blocks) * p.batch), kBwdThreads, DqCfg<D, VD>::kSmemBytes, stream>>>(p);
    e = cudaGetLastError();
    if (e != cudaSuccess) return e;
  }
  if (CL && !bwd_maps<T, D, VD, CL>(&p, a, kBN, kBM)) return cudaErrorInvalidValue;   // dK/dV kernels: resident keys
  if constexpr (D == 64 && VD == 64) {
    if (a.variant != 4) {
      auto kern = split ? bwd_dkdv_small_kernel<T, D, VD, true, CL> : bwd_dkdv_small_kernel<T, D, VD, false, CL>;
      cudaError_t e =
          plan::ensure_smem(kern, DkvSmallCfg<D, VD>::kSmemBytes);
      if (e != cudaSuccess) return e;
      p.n_blocks = (nk + kBM - 1) / kBM;
      ScopedKernel timed(CL ? (kBf16 ? "bwd_dkdv_bf16_sm100_2cta_cl" : "bwd_dkdv_f16_sm100_2cta_cl") : (kBf16 ? "bwd_dkdv_bf16_sm100_2cta" : "bwd_dkdv_f16_sm100_2cta"), stream);
      kern<<<unsigned(int64_t(p.n_blocks) * p.batch), kBwdThreads, DkvSmallCfg<D, VD>::kSmemBytes, stream>>>(p);
      return cudaGetLastError();
    }
  }
  {
    auto kern = split ? bwd_dkdv_kernel<T, D, VD, true, CL> : bwd_dkdv_kernel<T, D, VD, false, CL>;
    cudaError_t e =
        plan::ensure_smem(kern, DkvCfg<D, VD>::kSmemBytes);
    if (e != cudaSuccess) return e;
    p.n_blocks = (nk + kBM - 1) / kBM;
    ScopedKernel timed(CL ? (kBf16 ? "bwd_dkdv_bf16_sm100_cl" : "bwd_dkdv_f16_sm100_cl") : (kBf16 ? "bwd_dkdv_bf16_sm100" : "bwd_dkdv_f16_sm100"), stream);
    kern<<<unsigned(int64_t(p.n_blocks) * p.batch), kBwdThreads, DkvCfg<D, VD>::kSmemBytes, stream>>>(p);
    return cudaGetLastError();
  }
}

#ifdef FA_DBG_TIMELINE
extern "C" void fa_debug_set_buffer_bwd(void* buf) { cudaMemcpyToSymbol(g_dbg_bwd, &buf, sizeof(buf)); }
#endif

static int64_t pad8b(int64_t n) { return (n + 7) & ~int64_t(7); }
static size_t al256b(size_t v) { return (v + 255) & ~size_t(255); }

BwdLayout bwd_layout(const LaunchArgs& a) {
  BwdLayout w{};
  const int64_t nq = a.rule.q.total, nk = a.rule.k.total;
  // channel-last: the sequence is an outer dimension of the tensor maps - no pitch constraint, nothing to pack
  w.pack_q = a.layout == 0 && (nq % 8) != 0;
  w.pack_k = a.layout == 0 && (nk % 8) != 0;
  const int64_t qp = pad8b(nq), kp = pad8b(nk);
  size_t off = stats_bytes(a.batch, nq);
  auto take = [&off](size_t n) { size_t o = off; off += al256b(n); return o; };
  w.off_acc = off;
  if (a.d == 128 && a.variant != 4) take(size_t(a.batch) * 128 * qp * sizeof(float));
  if (w.pack_q) {
    w.off_q = take(size_t(a.batch) * a.d * qp * 2);
    w.off_do = take(size_t(a.batch) * a.v_d * qp * 2);
    w.off_dq = take(size_t(a.batch) * a.d * qp * 2);
  }
  if (w.pack_k) {
    w.off_k = take(size_t(a.batch) * a.d * kp * 2);
    w.off_v = take(size_t(a.batch) * a.v_d * kp * 2);
    w.off_dk = take(size_t(a.batch) * a.d * kp * 2);
    w.off_dv = take(size_t(a.batch) * a.v_d * kp * 2);
  }
  w.total = off;
  return w;
}

}  // namespace sm100

static bool aligned16b(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

bool sm100_f16_backward_supports(const LaunchArgs& a) {
  if (a.dtype != 0 && a.dtype != 3) return false;
  if (a.layout == 1) {
    if (a.heads < 1 || a.batch % a.heads) return false;
    if (a.d % 8 || a.v_d % 8) return false;   // strides of the 4-D tensor maps are multiples of 16 bytes
    if (!aligned16b(a.o)) return false;        // the statistics pass reads O, dO in 16-byte chunks
  } else if (a.layout != 0) {
    return false;
  }
  if (a.d < 1 || a.v_d < 1 || a.d > 128 || a.v_d > 128) return false;
  const int64_t nq = a.rule.q.total, nk = a.rule.k.total;
  const sm100::BwdLayout w = sm100::bwd_layout(a);
  if (!w.pack_q && (!aligned16b(a.q) || !aligned16b(a.d_o) || !aligned16b(a.d_q))) return false;
  if (!w.pack_k && (!aligned16b(a.k) || !aligned16b(a.v) || !aligned16b(a.d_k) || !aligned16b(a.d_v))) return false;
  if (!a.workspace || (reinterpret_cast<uintptr_t>(a.workspace) & 255) || a.workspace_bytes < w.total) return false;
  if (a.batch > 0x7fffffffLL) return false;
  if (((nq + 255) / 256) * a.batch > 0x7fffffffLL || ((nk + 127) / 128) * a.batch > 0x7fffffffLL) return false;
  // the per-CTA tile schedules hold 32 * kMaxTileWords streamed 64-wide tiles (keys in the dQ kernels, queries in the
  // dK/dV and fused kernels)
  if ((nk + 63) / 64 > 32 * sm100::kMaxTileWords || (nq + 63) / 64 > 32 * sm100::kMaxTileWords) return false;
  return true;
}

size_t sm100_f16_bwd_workspace_bytes(const LaunchArgs& a) { return sm100::bwd_layout(a).total; }

// fa_backward_accumulate: the fused head_dim-128 kernel on unpacked channel-first tensors (any gradient precision mode
// but "precise everywhere", which runs the two-kernel backward)
bool sm100_f16_backward_accumulate_supports(const LaunchArgs& a) {
  if (!sm100_f16_backward_supports(a)) return false;
  if (a.layout != 0 || a.d != 128 || (a.v_d != 128 && a.v_d != 64) || a.variant == 4 || a.grad_split == 1) return false;
  const int64_t nq = a.rule.q.total, nk = a.rule.k.total;
  if (nq % 8 || nk % 8) return false;                       // no pack pass in front of accumulators
  if (a.dq_fold < 1 || a.dq_fold > a.batch) return false;
  if ((reinterpret_cast<uintptr_t>(a.d_q) & 15) != 0) return false;
  return true;
}

template <typename T, bool CL>
static cudaError_t backward_dispatch_layout(const LaunchArgs& a, cudaStream_t stream) {
  const bool d_small = a.d <= 64, v_small = a.v_d <= 64;
  if (!d_small && !v_small) return sm100::launch_bwd<T, 128, 128, CL>(a, stream);
  if (d_small && v_small) return sm100::launch_bwd<T, 64, 64, CL>(a, stream);
  if (!d_small) return sm100::launch_bwd<T, 128, 64, CL>(a, stream);
  return sm100::launch_bwd<T, 64, 128, CL>(a, stream);
}
template <typename T>
static cudaError_t backward_dispatch_t(const LaunchArgs& a, cudaStream_t stream) {
  return a.layout == 1 ? backward_dispatch_layout<T, true>(a, stream) : backward_dispatch_layout<T, false>(a, stream);
}
static cudaError_t backward_dispatch(const LaunchArgs& a, cudaStream_t stream) {
  return a.dtype == 3 ? backward_dispatch_t<__nv_bfloat16>(a, stream) : backward_dispatch_t<__half>(a, stream);
}

cudaError_t sm100_f16_backward(const LaunchArgs& a0, cudaStream_t stream) {
  const sm100::BwdLayout w = sm100::bwd_layout(a0);
  LaunchArgs a = a0;
  a.prep_d_o = a0.d_o;   // the statistics pass reads the caller's dense O / dO
  if (!w.pack_q && !w.pack_k) return backward_dispatch(a, stream);
  char* ws = static_cast<char*>(a0.workspace);
  const int64_t nq = a.rule.q.total, nk = a.rule.k.total;
  cudaError_t e;
  if (w.pack_q) {
    a.q_pitch = sm100::pad8b(nq);
    if ((e = pack_rows(2, a0.q, ws + w.off_q, a.batch * a.d, nq, nq, a.q_pitch, stream)) != cudaSuccess) return e;
    if ((e = pack_rows(2, a0.d_o, ws + w.off_do, a.batch * a.v_d, nq, nq, a.q_pitch, stream)) != cudaSuccess) return e;
    a.q = ws + w.off_q;
    a.d_o = ws + w.off_do;
    a.d_q = ws + w.off_dq;
  }
  if (w.pack_k) {
    a.k_pitch = sm100::pad8b(nk);
    if ((e = pack_rows(2, a0.k, ws + w.off_k, a.batch * a.d, nk, nk, a.k_pitch, stream)) != cudaSuccess) return e;
    if ((e = pack_rows(2, a0.v, ws + w.off_v, a.batch * a.v_d, nk, nk, a.k_pitch, stream)) != cudaSuccess) return e;
    a.k = ws + w.off_k;
    a.v = ws + w.off_v;
    a.d_k = ws + w.off_dk;
    a.d_v = ws + w.off_dv;
  }
  if ((e = backward_dispatch(a, stream)) != cudaSuccess) return e;
  if (w.pack_q && (e = pack_rows(2, a.d_q, a0.d_q, a.batch * a.d, nq, a.q_pitch, nq, stream)) != cudaSuccess) return e;
  if (w.pack_k) {
    if ((e = pack_rows(2, a.d_k, a0.d_k, a.batch * a.d, nk, a.k_pitch, nk, stream)) != cudaSuccess) return e;
    if ((e = pack_rows(2, a.d_v, a0.d_v, a.batch * a.v_d, nk, a.k_pitch, nk, stream)) != cudaSuccess) return e;
  }
  return cudaSuccess;
}

}  // namespace fa
