// fa_fwd_f16_sm100.cu — Blackwell-native 16-bit (fp16 / bf16) forward: TMA -> swizzled smem -> tcgen05.mma with
// TMEM accumulators, warp-specialised (1 TMA producer warp, 1 MMA issuer warp, 2 softmax
// warpgroups that ping-pong over two 128-row Q tiles).
//
// Replaces the reference's ForwardImpl (flash_attention/kernel/flash_attention.cu:425-1077), a
// scalar-FMA kernel that walks K tiles in the outer loop and read-modify-writes O/l/m in HBM under a
// spin lock. Here each CTA owns 256 query rows of one batch element, streams only the K/V tiles the
// rule does not skip, keeps S/P and O in tensor memory and writes O, l, m exactly once.
//
// Layout facts this design leans on (channel-first tensors, sequence contiguous):
//   S = Q K^T : A = Q tile, B = K tile, both "MN-major" in shared memory (the 64-element swizzle
//               row runs along the sequence, 8 channels form one 1024-byte swizzle atom)
//   O = P V   : A = P (fp16 / bf16, written by the softmax warps into TMEM over S), B = V tile, K-major
// so no transposes are needed anywhere.
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

constexpr int kBlockM = 128;     // query rows per tile == TMEM lanes
constexpr int kQTiles = 2;       // Q tiles per CTA (ping-pong)
constexpr int kStages = 4;       // K/V ring depth (each stage holds one K or one V tile)
constexpr int kThreads = 384;    // 8 softmax warps + producer + mma + alloc + spare
constexpr float kLog2e = 1.4426950408889634f;
constexpr float kLn2 = 0.6931471805599453f;
constexpr float kRescaleThreshold = 8.0f;  // log2 units; lazy O rescale

struct alignas(64) FwdParams {
  CUtensorMap map_q, map_k, map_v, map_o;
  FaRule rule;
  float* l;
  void* m;         // T [batch][nq]
  int32_t nq, nk, n_qpairs;
  int32_t batch;
  int32_t heads;   // channel-last tensors: batch element = outer * heads + head
  float scale_log2;
};

#ifdef FA_DBG_TIMELINE
// developer-only (tools/timeline.py): clock64 stamps of CTA 0 -> g_dbg[role][j][event]
__device__ long long* g_dbg = nullptr;
#define FA_STAMP(role, j, ev)                                                     \
  do {                                                                            \
    if (g_dbg && blockIdx.x == 0 && (j) < 128) g_dbg[((role) * 128 + (j)) * 4 + (ev)] = clock64(); \
  } while (0)
#else
#define FA_STAMP(role, j, ev)
#endif

// BN = keys per streamed tile. 128 is the compute-bound configuration (one CTA per SM, 512 TMEM columns).
// BN = 64 with head_dim 64 needs 256 TMEM columns and ~66 KB of shared memory, so two CTAs share an SM
// (MINB = 2): short sequences and narrow windows are latency chains per CTA (prologue, 2-3 tiles, epilogue)
// and HBM-bound overall, and only a second resident CTA hides those chains.
// Softmax / MMA hand-off (round-2 A/B on B200, profiles/r2_fwd_variants.md; all variants bit-equal in O, l, m):
// the row max runs as four independent chains (a single chain is 63 dependent FMNMX3), and with 128-key tiles P is
// handed to the MMA warp in two halves, so P V of keys 0..63 runs while the exponentials of keys 64..127 are still
// being computed (C2 forward 1024 -> 1083 TFLOPS). Measured and removed (profiles/r2_fwd_variants.md): an event-driven
// issuer that also issued the upper half of the next Q K^T early (953), a 96 + 32 key hand-off (1059), exponentials
// issued against the previous reference max with the row max computed in their shadow (1069), an FA-3 style turn on
// the MUFU pipe between the two warpgroups (1080), 12.5 / 25 / 37.5 % of the exponentials as FMA-pipe polynomials
// (1076 / 1045 / 1004). The kernel runs under the board's power cap (1.58 GHz, sw_power_cap active for the whole
// run), so shortening stall chains buys nothing once the clock governor takes the cycles back: what counts is
// energy per tile.
template <int D, int VD, int BN>
struct FwdCfg {
  static constexpr bool kHalves = BN == 128;               // P handed over in two parts
  static constexpr int kSplitKs = 4;                       // first part: keys 0..63 (four K = 16 steps of P V)
  static constexpr int kCh = D > VD ? D : VD;
  static constexpr int kQTileBytes = kBlockM * kCh * 2;   // doubles as the O staging tile
  static constexpr int kStageBytes = BN * kCh * 2;
  static constexpr int kColO = kQTiles * BN;               // TMEM: S_i at i*BN (P aliased), O_i at kColO + i*VD
  static constexpr int kColsUsed = kColO + kQTiles * VD;
  static constexpr int kTmemCols = kColsUsed <= 256 ? 256 : 512;
  static constexpr int kBarOffset = kQTiles * kQTileBytes + kStages * kStageBytes;
  static constexpr int kNumBars = 2 + 2 * kStages + 2 + 2 + 2 + (kHalves ? 2 : 0);
  static constexpr int kSchedOffset = kBarOffset + kNumBars * 8 + 16;
  static constexpr int kSmemBytes = kSchedOffset + int(sizeof(TileSchedule)) + 1024;  // + alignment slack
};

// CL = the tensors are channel-last, [outer][sequence][heads][channels] (4-D tensor maps, one box = 64 channels of R
// positions of one head): the same tiles with positions and channels swapped, so every shared-memory operand flips
// between MN-major and K-major (sm100_ptx.cuh tile_desc) and O is staged row-major. Products, accumulation order and
// results are identical to the channel-first kernel's.
// T = __half or __nv_bfloat16: the element type of Q, K, V, O, m and of P in tensor memory.
template <typename T, int D, int VD, int BN, int MINB, bool CL>
__global__ void __launch_bounds__(kThreads, MINB) fwd_kernel(const __grid_constant__ FwdParams p) {
  using Cfg = FwdCfg<D, VD, BN>;
  constexpr int kBlockN = BN;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  const uint32_t q_smem = smem_base;
  const uint32_t kv_smem = smem_base + kQTiles * Cfg::kQTileBytes;
  const uint32_t bars = smem_base + Cfg::kBarOffset;
  const uint32_t bar_q_full = bars;                        // [2]
  const uint32_t bar_kv_full = bars + 16;                  // [kStages]
  const uint32_t bar_kv_empty = bar_kv_full + 8 * kStages; // [kStages]
  const uint32_t bar_s_full = bar_kv_empty + 8 * kStages;  // [2]
  const uint32_t bar_p_ready = bar_s_full + 16;            // [2]
  const uint32_t bar_o_final = bar_p_ready + 16;           // [2]
  const uint32_t bar_p_half = bar_o_final + 16;            // [2], two-halves hand-off only
  const uint32_t tmem_slot = bars + Cfg::kNumBars * 8;
  volatile uint32_t* tmem_slot_gen = reinterpret_cast<volatile uint32_t*>(smem_gen + Cfg::kBarOffset + Cfg::kNumBars * 8);

  const int warp = threadIdx.x >> 5;
  const FaRule& rule = p.rule;

  // CTAs of one batch element are adjacent (its K/V stay L2-resident while ~5 heads are in
  // flight); inside a head the heavy (late) query rows go first
  const int b = int(blockIdx.x / p.n_qpairs);
  const int head = CL ? b % p.heads : 0, outer = CL ? b / p.heads : b;
  (void)head; (void)outer;
  const int pair = p.n_qpairs - 1 - int(blockIdx.x % p.n_qpairs);
  const int q0 = pair * (kQTiles * kBlockM);
  const int q_hi = min(q0 + kQTiles * kBlockM, p.nq) - 1;
  int kt_first, kt_last;
  fa_k_tile_range(rule, q0, q_hi, kBlockN, &kt_first, &kt_last);
  TileSchedule* sched = reinterpret_cast<TileSchedule*>(smem_gen + Cfg::kSchedOffset);
  {
    const int lo[2] = {q0, q0 + kBlockM};
    const int hi[2] = {min(q0 + kBlockM, p.nq) - 1, min(q0 + 2 * kBlockM, p.nq) - 1};
    const bool valid[2] = {q0 < p.nq, q0 + kBlockM < p.nq};
    build_schedule(sched, rule, true, lo, hi, valid, 2, kt_first, kt_last, kBlockN, p.nk, kThreads / 32);
  }

  if (warp == 8) {
    if (elect_one()) {
      prefetch_tensormap(&p.map_q);
      prefetch_tensormap(&p.map_k);
      prefetch_tensormap(&p.map_v);
      prefetch_tensormap(&p.map_o);
    }
  } else if (warp == 9) {
    if (elect_one()) {
      for (int i = 0; i < 2; ++i) {
        mbar_init(bar_q_full + 8 * i, 1);
        mbar_init(bar_s_full + 8 * i, 1);
        mbar_init(bar_p_ready + 8 * i, kBlockM);
        mbar_init(bar_o_final + 8 * i, 1);
        if constexpr (Cfg::kHalves) mbar_init(bar_p_half + 8 * i, kBlockM);
      }
      for (int s = 0; s < kStages; ++s) {
        mbar_init(bar_kv_full + 8 * s, 1);
        mbar_init(bar_kv_empty + 8 * s, 1);
      }
      fence_barrier_init();
    }
  } else if (warp == 10) {
    tmem_alloc(tmem_slot, Cfg::kTmemCols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_gen;

  if (warp >= 8) {
    if constexpr (MINB == 1)
      setmaxnreg_dec<56>();
    else
      setmaxnreg_dec<32>();
    if (warp == 8) {
      // ===================== TMA producer =====================
      if (elect_one()) {
        for (int i = 0; i < kQTiles; ++i) {
          mbar_arrive_expect_tx(bar_q_full + 8 * i, kBlockM * D * 2);
          if constexpr (CL) {
            for (int c = 0; c < D / 64; ++c)
              tma_load_cl(q_smem + i * Cfg::kQTileBytes + c * (kBlockM * 128), &p.map_q, bar_q_full + 8 * i, c * 64,
                          head, q0 + i * kBlockM, outer);
          } else {
            for (int h = 0; h < 2; ++h)
              tma_load_bc(q_smem + i * Cfg::kQTileBytes + h * (D * 128), &p.map_q, bar_q_full + 8 * i,
                          q0 + i * kBlockM + h * 64, b);
          }
        }
        int t = 0;
        TileIter it;
        it.init(sched, 2, kt_first, kt_last);
        int kt, tw, tb;
        while (it.next(&kt, &tw, &tb)) {
          {
            const int s = t % kStages, u = t / kStages;
            mbar_wait(bar_kv_empty + 8 * s, (u & 1) ^ 1);
            mbar_arrive_expect_tx(bar_kv_full + 8 * s, kBlockN * D * 2);
            if constexpr (CL) {
              for (int c = 0; c < D / 64; ++c)
                tma_load_cl(kv_smem + s * Cfg::kStageBytes + c * (kBlockN * 128), &p.map_k, bar_kv_full + 8 * s, c * 64,
                            head, kt * kBlockN, outer);
            } else {
              for (int h = 0; h < kBlockN / 64; ++h)
                tma_load_bc(kv_smem + s * Cfg::kStageBytes + h * (D * 128), &p.map_k, bar_kv_full + 8 * s,
                            kt * kBlockN + h * 64, b);
            }
            ++t;
          }
          {
            const int s = t % kStages, u = t / kStages;
            mbar_wait(bar_kv_empty + 8 * s, (u & 1) ^ 1);
            mbar_arrive_expect_tx(bar_kv_full + 8 * s, kBlockN * VD * 2);
            if constexpr (CL) {
              for (int c = 0; c < VD / 64; ++c)
                tma_load_cl(kv_smem + s * Cfg::kStageBytes + c * (kBlockN * 128), &p.map_v, bar_kv_full + 8 * s, c * 64,
                            head, kt * kBlockN, outer);
            } else {
              for (int h = 0; h < kBlockN / 64; ++h)
                tma_load_bc(kv_smem + s * Cfg::kStageBytes + h * (VD * 128), &p.map_v, bar_kv_full + 8 * s,
                            kt * kBlockN + h * 64, b);
            }
            ++t;
          }
        }
      }
    } else if (warp == 9) {
      // ===================== MMA issuer =====================
      if (elect_one()) {
        TileIter it;
        it.init(sched, 2, kt_first, kt_last);
        const int n = it.count();
        constexpr uint32_t idesc_qk = idesc_16<T>(kBlockM, kBlockN, tile_mn_major<CL>(true), tile_mn_major<CL>(true));
        constexpr uint32_t idesc_pv = idesc_16<T>(kBlockM, VD, false, tile_mn_major<CL>(false));
        auto issue_qk = [&](int i, int stage) {
          const uint32_t a0 = q_smem + i * Cfg::kQTileBytes;
          const uint32_t b0 = kv_smem + stage * Cfg::kStageBytes;
#pragma unroll
          for (int ks = 0; ks < D / 16; ++ks) {
            // channel-first: MN-major SW128, 16 channels = two 1024-byte atoms, LBO = next 64 rows (next TMA box)
            const uint64_t da = tile_desc<CL>(a0, ks, kBlockM, D, true);
            const uint64_t db = tile_desc<CL>(b0, ks, kBlockN, D, true);
            mma_ss(tmem_base + i * kBlockN, da, db, idesc_qk, ks > 0);
          }
        };
        // first part: keys [0, 16 * kSplitKs), handed over while the last exponentials are still running; second part: the rest
        auto issue_pv_half = [&](int i, int stage, bool accumulate, int half) {
          const uint32_t b0 = kv_smem + stage * Cfg::kStageBytes;
#pragma unroll
          for (int ks = half * Cfg::kSplitKs; ks < (half ? kBlockN / 16 : Cfg::kSplitKs); ++ks) {
            const uint64_t db = tile_desc<CL>(b0, ks, kBlockN, VD, false);
            mma_ts(tmem_base + Cfg::kColO + i * VD, tmem_base + i * kBlockN + ks * 8, db, idesc_pv,
                   (accumulate || ks > 0) ? 1u : 0u);
          }
        };
        auto issue_pv = [&](int i, int stage, bool accumulate) {
          const uint32_t b0 = kv_smem + stage * Cfg::kStageBytes;
#pragma unroll
          for (int ks = 0; ks < kBlockN / 16; ++ks) {
            // channel-first: K-major SW128, 16 keys = 32 bytes inside the 128-byte row; second box after 64 keys
            const uint64_t db = tile_desc<CL>(b0, ks, kBlockN, VD, false);
            mma_ts(tmem_base + Cfg::kColO + i * VD, tmem_base + i * kBlockN + ks * 8, db, idesc_pv,
                   (accumulate || ks > 0) ? 1u : 0u);
          }
        };
        if (n > 0) {
          mbar_wait(bar_kv_full + 0, 0);
          for (int i = 0; i < kQTiles; ++i) {
            mbar_wait(bar_q_full + 8 * i, 0);
            tc_fence_after();
            issue_qk(i, 0);
            mma_commit(bar_s_full + 8 * i);
          }
          mma_commit(bar_kv_empty + 0);
          for (int j = 0; j < n; ++j) {
            const int tv = 2 * j + 1, sv = tv % kStages;
            const int tk = 2 * j + 2, sk = tk % kStages;
            mbar_wait(bar_kv_full + 8 * sv, (tv / kStages) & 1);
            for (int i = 0; i < kQTiles; ++i) {
              if constexpr (Cfg::kHalves) {
                mbar_wait(bar_p_half + 8 * i, j & 1);
                tc_fence_after();
                issue_pv_half(i, sv, j > 0, 0);
                mbar_wait(bar_p_ready + 8 * i, j & 1);
                tc_fence_after();
                FA_STAMP(2 + i, j, 0);
                issue_pv_half(i, sv, true, 1);
              } else {
                mbar_wait(bar_p_ready + 8 * i, j & 1);
                tc_fence_after();
                FA_STAMP(2 + i, j, 0);
                issue_pv(i, sv, j > 0);
              }
              if (i == kQTiles - 1) mma_commit(bar_kv_empty + 8 * sv);
              if (j + 1 < n) {
                if (i == 0) {
                  mbar_wait(bar_kv_full + 8 * sk, (tk / kStages) & 1);
                  tc_fence_after();
                }
                issue_qk(i, sk);
                mma_commit(bar_s_full + 8 * i);
                FA_STAMP(2 + i, j, 1);
                if (i == kQTiles - 1) mma_commit(bar_kv_empty + 8 * sk);
              } else {
                mma_commit(bar_o_final + 8 * i);
              }
            }
          }
        }
      }
    }
  } else {
    // ===================== softmax warpgroups =====================
    if constexpr (MINB == 1)
      setmaxnreg_inc<224>();
    else
      setmaxnreg_inc<104>();
    const int i = warp >> 2;                    // which Q tile
    const int r = threadIdx.x & 127;            // row inside the tile
    const uint32_t lane_addr = uint32_t((warp & 3) * 32) << 16;
    const uint32_t t_s = tmem_base + lane_addr + i * kBlockN;
    const uint32_t t_o = tmem_base + lane_addr + Cfg::kColO + i * VD;
    const int tq0 = q0 + i * kBlockM;
    const int tq_hi = min(tq0 + kBlockM, p.nq) - 1;
    const bool tile_valid = tq0 < p.nq;
    const int qi = tq0 + r;
    const bool q_valid = qi < p.nq;
    const FaPos qpos = fa_pos(rule, rule.q, min(qi, p.nq - 1));
    const float scale_log2 = p.scale_log2;
    const float NEG_INF = __int_as_float(0xff800000);
    float m_ref = NEG_INF;   // running reference max (log2 units) the accumulators are scaled to
    float m_true = NEG_INF;  // true running max (log2 units)
    float l_sum = 0.f;
    int j = 0;
    TileIter it;
    it.init(sched, 2, kt_first, kt_last);
    int kt, tw, tb;
    while (it.next(&kt, &tw, &tb)) {
      const int k0 = kt * kBlockN;
      const int k_hi = min(k0 + kBlockN, p.nk) - 1;
      const int cls = it.cls(i, tw, tb);
      const bool ragged = k0 + kBlockN > p.nk;
      mbar_wait(bar_s_full + 8 * i, j & 1);
      tc_fence_after();
      if (r == 0) FA_STAMP(i, j, 0);
      // attended-column bitmask of this row for this tile (only built for PARTIAL / ragged tiles).
      // Built BEFORE the TMEM load is issued: nothing that could make the compiler move or spill the
      // destination registers (e.g. the out-of-line mask builder) may sit between tcgen05.ld and
      // tcgen05.wait::ld.
      const bool masked = cls != FA_TILE_FULL || ragged;
      uint32_t okm[kBlockN / 32] = {};
      if (masked && cls != FA_TILE_SKIP) {
        const int nvalid = k_hi - k0 + 1;
        if (rule.dims == 1 && rule.rule != 2) {
          int lo, hi;
          interval_1d(rule, true, qpos, k0, nvalid, &lo, &hi);
#pragma unroll
          for (int c = 0; c < kBlockN / 32; ++c) okm[c] = interval_bits32(lo, hi, 32 * c);
        } else {
#pragma unroll
          for (int c = 0; c < kBlockN / 32; ++c) okm[c] = tile_mask32(rule, true, qpos, k0, 32 * c, nvalid);
        }
      }
      // S row -> registers (one row per thread)
      float s[kBlockN];
#pragma unroll
      for (int c = 0; c < kBlockN / 32; ++c) tmem_ld32f(t_s + c * 32, &s[c * 32]);
      tmem_wait_ld();
      if (masked) {
#pragma unroll
        for (int c = 0; c < kBlockN; ++c) s[c] = (okm[c >> 5] >> (c & 31)) & 1u ? s[c] : NEG_INF;
      }
      if (r == 0) FA_STAMP(i, j, 1);
      // row max as four independent chains (each still fuses into 3-input max instructions)
      auto row_max = [&]() {
        float m4[4] = {s[0], s[1], s[2], s[3]};
#pragma unroll
        for (int c = 4; c + 8 <= kBlockN; c += 8) {
#pragma unroll
          for (int e = 0; e < 4; ++e) m4[e] = fmaxf(fmaxf(m4[e], s[c + e]), s[c + 4 + e]);
        }
#pragma unroll
        for (int e = 0; e < 4; ++e) m4[e] = fmaxf(m4[e], s[kBlockN - 4 + e]);
        return fmaxf(fmaxf(m4[0], m4[1]), fmaxf(m4[2], m4[3]));
      };
      uint32_t pk0[16], pk1[16];
      const float mx2 = row_max() * scale_log2;   // -inf stays -inf (scale > 0)
      m_true = fmaxf(m_true, mx2);
      if (j == 0) {
        m_ref = mx2;
      } else {
        const bool need = mx2 > m_ref + kRescaleThreshold;
        if (__any_sync(0xffffffffu, need)) {
          const float m_new = fmaxf(m_ref, mx2);
          const float alpha = (m_new == NEG_INF) ? 1.f : ex2(m_ref - m_new);
          m_ref = m_new;
          l_sum *= alpha;
#pragma unroll 1
          for (int c = 0; c < VD / 32; ++c) {
            float o[32];
            tmem_ld32f(t_o + c * 32, o);
            tmem_wait_ld();
#pragma unroll
            for (int e = 0; e < 32; ++e) o[e] *= alpha;
            tmem_st32f(t_o + c * 32, o);
          }
        }
      }
      const float m_use = (m_ref == NEG_INF) ? 0.f : m_ref;
      float sum0 = 0.f, sum1 = 0.f;
      auto exp_cols = [&](int c0, int n, uint32_t* pk) {   // columns [c0, c0 + n) -> pairs of T
#pragma unroll
        for (int e = 0; e < n; e += 2) {
          const float p0 = ex2(fmaf(s[c0 + e], scale_log2, -m_use));
          const float p1 = ex2(fmaf(s[c0 + e + 1], scale_log2, -m_use));
          sum0 += p0;
          sum1 += p1;
          pk[e >> 1] = pack2<T>(p0, p1);
        }
      };
      // P = exp2(S*scale*log2e - m) -> pairs of T written over S, 32 columns at a time
      if constexpr (Cfg::kHalves) {
        exp_cols(0, 32, pk0);
        tmem_st16(t_s + 0, pk0);
        exp_cols(32, 32, pk1);
        tmem_st16(t_s + 16, pk1);
        exp_cols(64, 32, pk0);        // the stores of the first half complete under these exponentials
        tmem_wait_st();
        tc_fence_before();
        mbar_arrive(bar_p_half + 8 * i);   // keys 0..63 of P are in TMEM: P V can start on them
        tmem_st16(t_s + 32, pk0);
        exp_cols(96, 32, pk1);
        tmem_st16(t_s + 48, pk1);
      } else {
#pragma unroll
        for (int c = 0; c < kBlockN / 32; ++c) {
          exp_cols(c * 32, 32, pk0);
          tmem_st16(t_s + c * 16, pk0);
        }
      }
      l_sum += sum0 + sum1;
      if (r == 0) FA_STAMP(i, j, 2);
      tmem_wait_st();
      tc_fence_before();
      mbar_arrive(bar_p_ready + 8 * i);
      if (r == 0) FA_STAMP(i, j, 3);
      ++j;
    }

    // ---- epilogue: O = acc / l -> T -> smem [VD][64] x2 -> TMA store; l, m -> global ----
    uint8_t* stage_gen = smem_gen + i * Cfg::kQTileBytes;
    T* stage_h = reinterpret_cast<T*>(stage_gen) + (r >> 6) * (VD * 64) + (r & 63);
    if (j > 0) {
      mbar_wait(bar_o_final + 8 * i, 0);
      tc_fence_after();
      const float inv = l_sum > 0.f ? 1.f / l_sum : 0.f;
#pragma unroll
      for (int c = 0; c < VD / 32; ++c) {
        float o[32];
        tmem_ld32f(t_o + c * 32, o);
        tmem_wait_ld();
        if constexpr (CL) {
#pragma unroll
          for (int e = 0; e < 32; e += 8) {
            uint4 w;
            w.x = pack2<T>(o[e] * inv, o[e + 1] * inv);       // inv = 0 for rows without keys
            w.y = pack2<T>(o[e + 2] * inv, o[e + 3] * inv);
            w.z = pack2<T>(o[e + 4] * inv, o[e + 5] * inv);
            w.w = pack2<T>(o[e + 6] * inv, o[e + 7] * inv);
            *reinterpret_cast<uint4*>(stage_gen + cl_chunk_offset(r, c * 32 + e, kBlockM)) = w;
          }
        } else {
#pragma unroll
          for (int e = 0; e < 32; ++e) stage_h[(c * 32 + e) * 64] = from_acc<T>(l_sum > 0.f ? o[e] * inv : 0.f);
        }
      }
    } else {
      // no key tile survives for this CTA: wait for Q to land before reusing its buffer
      mbar_wait(bar_q_full + 8 * i, 0);
      if constexpr (CL) {
#pragma unroll 4
        for (int c = 0; c < VD; c += 8)
          *reinterpret_cast<uint4*>(stage_gen + cl_chunk_offset(r, c, kBlockM)) = make_uint4(0, 0, 0, 0);
      } else {
#pragma unroll 8
        for (int c = 0; c < VD; ++c) stage_h[c * 64] = from_acc<T>(0.f);
      }
    }
    if (q_valid) {
      const int64_t idx = int64_t(b) * p.nq + qi;
      T* m = static_cast<T*>(p.m);
      if (l_sum > 0.f) {
        const T m_h = from_acc<T>(m_true * kLn2);
        m[idx] = m_h;
        p.l[idx] = l_sum * ex2(m_ref - to_acc<float>(m_h) * kLog2e);
      } else {
        m[idx] = sentinel<T>();
        p.l[idx] = 0.f;
      }
    }
    fence_proxy_async_smem();
    named_bar_sync(1 + i, kBlockM);
    if (r == 0 && tile_valid) {
      if constexpr (CL) {
        for (int c = 0; c < VD / 64; ++c)
          tma_store_cl(&p.map_o, q_smem + i * Cfg::kQTileBytes + c * (kBlockM * 128), c * 64, head, tq0, outer);
      } else {
        for (int h = 0; h < 2; ++h)
          if (tq0 + h * 64 < p.nq)
            tma_store_bc(&p.map_o, q_smem + i * Cfg::kQTileBytes + h * (VD * 128), tq0 + h * 64, b);
      }
      tma_store_commit();
      tma_store_wait_read();
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 10) {
    tc_fence_after();
    tmem_dealloc(tmem_base, Cfg::kTmemCols);
  }
}

// ---- host side ---------------------------------------------------------------------------------
// 2-D view [rows = batch*channels][cols = sequence] of a channel-first fp16 tensor (the fp32 families' bf16 / workspace
// tensors are described this way)
bool make_map_2d(CUtensorMap* map, const void* base, int64_t rows, int64_t cols, int box_cols, int box_rows,
                 bool swizzle128) {
  const uint64_t gdim[2] = {uint64_t(cols), uint64_t(rows)};
  const uint64_t gstride[1] = {uint64_t(cols) * 2};
  const uint32_t box[2] = {uint32_t(box_cols), uint32_t(box_rows)};
  return plan::tensor_map(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, base, gdim, gstride, box,
                          swizzle128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE);
}

// 3-D view [batch][channels][sequence] of a channel-first 16-bit tensor (`pitch` elements between channel rows): the box
// is 64 positions x box_rows channels of one batch element; channels past `channels` are zero-filled / clipped.
bool make_map_3d(CUtensorMap* map, const void* base, int64_t batch, int64_t channels, int64_t seq, int64_t pitch,
                 int box_rows, bool swizzle128, CUtensorMapDataType dtype) {
  const uint64_t gdim[3] = {uint64_t(seq), uint64_t(channels), uint64_t(batch)};
  const uint64_t gstride[2] = {uint64_t(pitch) * 2, uint64_t(pitch) * 2 * uint64_t(channels)};
  const uint32_t box[3] = {64u, uint32_t(box_rows), 1u};
  return plan::tensor_map(map, dtype, 3, base, gdim, gstride, box,
                          swizzle128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE);
}

// 4-D view [outer][sequence][heads][channels] of a channel-last 16-bit tensor: the box is 64 channels x box_rows positions
// of one head (one 128-byte-row slab of a tile); channels past `channels` and positions past `seq` are zero-filled on
// loads and clipped on stores.
bool make_map_cl(CUtensorMap* map, const void* base, int64_t outer, int64_t heads, int64_t channels, int64_t seq,
                 int box_rows, CUtensorMapDataType dtype) {
  const uint64_t gdim[4] = {uint64_t(channels), uint64_t(heads), uint64_t(seq), uint64_t(outer)};
  const uint64_t gstride[3] = {uint64_t(channels) * 2, uint64_t(channels) * 2 * uint64_t(heads),
                               uint64_t(channels) * 2 * uint64_t(heads) * uint64_t(seq)};
  const uint32_t box[4] = {64u, 1u, uint32_t(box_rows), 1u};
  return plan::tensor_map(map, dtype, 4, base, gdim, gstride, box, CU_TENSOR_MAP_SWIZZLE_128B);
}

template <typename T, int D, int VD, int BN, int MINB, bool CL>
cudaError_t launch_fwd(const LaunchArgs& a, cudaStream_t stream) {
  using Cfg = FwdCfg<D, VD, BN>;
  constexpr CUtensorMapDataType dt = Elt16<T>::kTmaType;
  constexpr bool bf16 = std::is_same<T, __nv_bfloat16>::value;
  FwdParams p;
  const int nq = a.rule.q.total, nk = a.rule.k.total;
  // D, VD are the kernel's padded channel counts (a.d <= D, a.v_d <= VD)
  if constexpr (CL) {
    const int64_t heads = a.heads > 0 ? a.heads : 1, outer = a.batch / heads;
    if (!make_map_cl(&p.map_q, a.q, outer, heads, a.d, nq, kBlockM, dt) ||
        !make_map_cl(&p.map_k, a.k, outer, heads, a.d, nk, BN, dt) ||
        !make_map_cl(&p.map_v, a.v, outer, heads, a.v_d, nk, BN, dt) ||
        !make_map_cl(&p.map_o, a.o, outer, heads, a.v_d, nq, kBlockM, dt))
      return cudaErrorInvalidValue;
    p.heads = int32_t(heads);
  } else {
    const int64_t qp = a.q_pitch ? a.q_pitch : nq, kp = a.k_pitch ? a.k_pitch : nk;
    if (!make_map_3d(&p.map_q, a.q, a.batch, a.d, nq, qp, D, true, dt) ||
        !make_map_3d(&p.map_k, a.k, a.batch, a.d, nk, kp, D, true, dt) ||
        !make_map_3d(&p.map_v, a.v, a.batch, a.v_d, nk, kp, VD, true, dt) ||
        !make_map_3d(&p.map_o, a.o, a.batch, a.v_d, nq, qp, VD, false, dt))
      return cudaErrorInvalidValue;
    p.heads = 1;
  }
  p.rule = a.rule;
  p.l = (float*)a.l;
  p.m = a.m;
  p.nq = nq;
  p.nk = nk;
  p.n_qpairs = (nq + kQTiles * kBlockM - 1) / (kQTiles * kBlockM);
  p.batch = int32_t(a.batch);
  p.scale_log2 = kLog2e / sqrtf(float(a.d));
  auto kern = fwd_kernel<T, D, VD, BN, MINB, CL>;
  cudaError_t e = plan::ensure_smem(kern, Cfg::kSmemBytes);
  if (e != cudaSuccess) return e;
  const char* name = bf16 ? (CL ? (BN == 128 ? "fwd_bf16_sm100_cl" : "fwd_bf16_sm100_n64_cl")
                                 : (BN == 128 ? "fwd_bf16_sm100" : "fwd_bf16_sm100_n64"))
                          : (CL ? (BN == 128 ? "fwd_f16_sm100_cl" : "fwd_f16_sm100_n64_cl")
                                : (BN == 128 ? "fwd_f16_sm100" : "fwd_f16_sm100_n64"));
  ScopedKernel timed(name, stream);
  kern<<<unsigned(int64_t(p.n_qpairs) * p.batch), kThreads, Cfg::kSmemBytes, stream>>>(p);
  return cudaGetLastError();
}

#ifdef FA_DBG_TIMELINE
extern "C" void fa_debug_set_buffer(void* buf) { cudaMemcpyToSymbol(g_dbg, &buf, sizeof(buf)); }
#endif
}  // namespace sm100

static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }
static int64_t pad8(int64_t n) { return (n + 7) & ~int64_t(7); }
static size_t al256(size_t v) { return (v + 255) & ~size_t(255); }

// Pitch-padded copies in the workspace for lengths that are not multiples of 8 halves (fa_pack.cu).
struct FwdPack {
  bool q, k;
  size_t off_q, off_k, off_v, off_o, total;
};
static FwdPack fwd_pack_layout(const LaunchArgs& a) {
  FwdPack w{};
  const int64_t nq = a.rule.q.total, nk = a.rule.k.total;
  if (a.layout == 1) return w;   // channel-last: the sequence is an outer dimension of the tensor maps, any length
  w.q = (nq % 8) != 0;
  w.k = (nk % 8) != 0;
  size_t off = 0;
  auto take = [&off](size_t n) { size_t o = off; off += al256(n); return o; };
  if (w.q) {
    w.off_q = take(size_t(a.batch) * a.d * pad8(nq) * 2);
    w.off_o = take(size_t(a.batch) * a.v_d * pad8(nq) * 2);
  }
  if (w.k) {
    w.off_k = take(size_t(a.batch) * a.d * pad8(nk) * 2);
    w.off_v = take(size_t(a.batch) * a.v_d * pad8(nk) * 2);
  }
  w.total = off;
  return w;
}

// Any channel counts up to 128 (zero-filled up to the kernel's 64 / 128 through the 3-D tensor maps) and any sequence
// lengths (packed to a 16-byte pitch when needed): the shapes the reference's own tests draw (tests/test_1d.py:57-66,
// test_2d.py:85-94: channels 8..32, arbitrary even lengths) run on the tensor cores.
bool sm100_f16_forward_supports(const LaunchArgs& a) {
  if ((a.dtype != 0 && a.dtype != 3) || a.accumulate) return false;
  if (a.d < 1 || a.v_d < 1 || a.d > 128 || a.v_d > 128) return false;
  const int64_t nq = a.rule.q.total, nk = a.rule.k.total;
  const FwdPack w = fwd_pack_layout(a);
  if (a.layout == 1) {
    // channel-last: the strides between heads / positions are channels * 2 and heads * channels * 2 bytes
    if (a.heads < 1 || a.batch % a.heads) return false;
    if (a.d % 8 || a.v_d % 8) return false;
  } else if (a.layout != 0) {
    return false;
  }
  // TMA: base addresses and row pitches must be multiples of 16 bytes; a side whose length is not a multiple of 8 is
  // copied into the workspace, a misaligned base with an aligned length is left to the generic kernels
  if (!w.q && (!aligned16(a.q) || !aligned16(a.o))) return false;
  if (!w.k && (!aligned16(a.k) || !aligned16(a.v))) return false;
  if (w.total && (!a.workspace || (reinterpret_cast<uintptr_t>(a.workspace) & 255) || a.workspace_bytes < w.total))
    return false;
  if (a.batch > 0x7fffffffLL) return false;
  const int64_t pairs = (nq + 255) / 256;
  if (pairs * a.batch > 0x7fffffffLL) return false;
  // the per-CTA tile schedule holds 32 * kMaxTileWords streamed tiles (64-key tiles for head_dim <= 64, else 128-key)
  const int64_t tile = (a.d <= 64 && a.v_d <= 64 && a.variant != 5) ? 64 : 128;
  if ((nk + tile - 1) / tile > 32 * sm100::kMaxTileWords) return false;
  return true;
}

size_t sm100_f16_bwd_workspace_bytes(const LaunchArgs& a);  // fa_bwd_f16_sm100.cu
size_t sm100_f16_workspace_bytes(const LaunchArgs& a, bool backward) {
  if (a.d > 128 || a.v_d > 128) return 0;
  return backward ? sm100_f16_bwd_workspace_bytes(a) : fwd_pack_layout(a).total;
}

// head_dim <= 64: the 64-key / two-CTAs-per-SM configuration is faster on every workload measured (S1 1.01 -> 0.67 ms,
// S2 3.95 -> 2.01 ms, C3 0.84 -> 0.51 ms, C4 0.86 -> 0.73 ms; profiles/r1_short_sequences.md); override 5 keeps the
// 128-key / one-CTA configuration reachable for A/B runs.
template <typename T, bool CL>
static cudaError_t forward_dispatch_layout(const LaunchArgs& a, cudaStream_t stream) {
  const bool d_small = a.d <= 64, v_small = a.v_d <= 64;
  if (!d_small && !v_small) return sm100::launch_fwd<T, 128, 128, 128, 1, CL>(a, stream);
  if (d_small && v_small) {
    if (a.variant != 5) return sm100::launch_fwd<T, 64, 64, 64, 2, CL>(a, stream);
    return sm100::launch_fwd<T, 64, 64, 128, 1, CL>(a, stream);
  }
  if (!d_small) return sm100::launch_fwd<T, 128, 64, 128, 1, CL>(a, stream);
  return sm100::launch_fwd<T, 64, 128, 128, 1, CL>(a, stream);
}
template <typename T>
static cudaError_t forward_dispatch_t(const LaunchArgs& a, cudaStream_t stream) {
  return a.layout == 1 ? forward_dispatch_layout<T, true>(a, stream) : forward_dispatch_layout<T, false>(a, stream);
}
static cudaError_t forward_dispatch(const LaunchArgs& a, cudaStream_t stream) {
  return a.dtype == 3 ? forward_dispatch_t<__nv_bfloat16>(a, stream) : forward_dispatch_t<__half>(a, stream);
}

cudaError_t sm100_f16_forward(const LaunchArgs& a0, cudaStream_t stream) {
  const FwdPack w = fwd_pack_layout(a0);
  if (!w.total) return forward_dispatch(a0, stream);
  LaunchArgs a = a0;
  char* ws = static_cast<char*>(a0.workspace);
  const int64_t nq = a.rule.q.total, nk = a.rule.k.total;
  cudaError_t e;
  if (w.q) {
    a.q_pitch = pad8(nq);
    if ((e = pack_rows(2, a0.q, ws + w.off_q, a.batch * a.d, nq, nq, a.q_pitch, stream)) != cudaSuccess) return e;
    a.q = ws + w.off_q;
    a.o = ws + w.off_o;
  }
  if (w.k) {
    a.k_pitch = pad8(nk);
    if ((e = pack_rows(2, a0.k, ws + w.off_k, a.batch * a.d, nk, nk, a.k_pitch, stream)) != cudaSuccess) return e;
    if ((e = pack_rows(2, a0.v, ws + w.off_v, a.batch * a.v_d, nk, nk, a.k_pitch, stream)) != cudaSuccess) return e;
    a.k = ws + w.off_k;
    a.v = ws + w.off_v;
  }
  if ((e = forward_dispatch(a, stream)) != cudaSuccess) return e;
  if (w.q) return pack_rows(2, ws + w.off_o, a0.o, a.batch * a.v_d, nq, a.q_pitch, nq, stream);
  return cudaSuccess;
}

}  // namespace fa
