// sm100_ptx.cuh — thin inline-PTX wrappers for the Blackwell (sm_100a) primitives the
// attention kernels use: mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (alloc / mma / commit /
// ld / st / fences), setmaxnreg, named barriers. Hand-written; no CuTe / CUTLASS.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdint.h>

#include "fa_common.cuh"

namespace fa {
namespace ptx {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred P;\n\t.reg .b32 R;\n\t"
      "elect.sync R|P, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t}"
      : "=r"(pred));
  return pred != 0;
}

// ---- mbarrier -------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred P;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {
  }
}

// ---- TMA ------------------------------------------------------------------------------------
__device__ __forceinline__ void prefetch_tensormap(const void* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(map)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t smem_dst, const void* map, uint32_t bar, int32_t x,
                                            int32_t y) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(x), "r"(y)
      : "memory");
}
__device__ __forceinline__ void tma_store_2d(const void* map, uint32_t smem_src, int32_t x, int32_t y) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(map)),
               "r"(smem_src), "r"(x), "r"(y)
               : "memory");
}
// Channel-first tensors are described to TMA as 3-D [batch][channels][sequence] (fa::sm100::make_map_3d): the box spans
// 64 sequence positions x the kernel's padded channel count of ONE batch element, so channels beyond the tensor's own
// count are zero-filled on loads and clipped on stores instead of reading / writing the next batch element.
__device__ __forceinline__ void tma_load_bc(uint32_t smem_dst, const void* map, uint32_t bar, int32_t x, int32_t b) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(smem_dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(x), "r"(0), "r"(b)
      : "memory");
}
__device__ __forceinline__ void tma_store_bc(const void* map, uint32_t smem_src, int32_t x, int32_t b) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(map)),
               "r"(smem_src), "r"(x), "r"(0), "r"(b)
               : "memory");
}
// 4-D tile copies of channel-last tensors [outer][sequence][heads][channels]: coordinates (channel, head, position,
// outer); the box is 64 channels x R positions of one head, i.e. one 128-byte-row slab of a tile in shared memory.
__device__ __forceinline__ void tma_load_cl(uint32_t smem_dst, const void* map, uint32_t bar, int32_t c, int32_t h,
                                            int32_t s, int32_t b) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(smem_dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c), "r"(h), "r"(s), "r"(b)
      : "memory");
}
__device__ __forceinline__ void tma_store_cl(const void* map, uint32_t smem_src, int32_t c, int32_t h, int32_t s,
                                             int32_t b) {
  asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(map)),
               "r"(smem_src), "r"(c), "r"(h), "r"(s), "r"(b)
               : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// shared-memory source of every committed bulk store has been read (enough before the CTA reuses the tile or exits;
// the global writes complete on their own before the grid does)
__device__ __forceinline__ void tma_store_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}
__device__ __forceinline__ void tma_store_wait_all() {
  asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}
// generic-proxy smem writes -> visible to the async proxy (TMA store / UMMA operand reads)
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

// ---- tcgen05 --------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t smem_result_addr, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_result_addr),
               "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
// D[tmem] (+)= A[smem] * B[smem]
__device__ __forceinline__ void mma_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                       uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem]
__device__ __forceinline__ void mma_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc,
                                       uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}" ::"r"(d_tmem),
      "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// TF32 variants (32-bit containers, 10-bit mantissa used; K = 8 per instruction)
__device__ __forceinline__ void mma_ss_tf32(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                            uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void mma_ts_tf32(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc,
                                            uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}" ::"r"(d_tmem),
      "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrive on an mbarrier once every previously issued tcgen05 op of this thread has completed
__device__ __forceinline__ void mma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar)
               : "memory");
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// 32 lanes x 32 consecutive 32-bit columns; thread i of the warp <-> TMEM lane (lane_base + i)
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]),
        "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]),
        "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld32f(uint32_t taddr, float* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=f"(r[0]), "=f"(r[1]), "=f"(r[2]), "=f"(r[3]), "=f"(r[4]), "=f"(r[5]), "=f"(r[6]), "=f"(r[7]),
        "=f"(r[8]), "=f"(r[9]), "=f"(r[10]), "=f"(r[11]), "=f"(r[12]), "=f"(r[13]), "=f"(r[14]), "=f"(r[15]),
        "=f"(r[16]), "=f"(r[17]), "=f"(r[18]), "=f"(r[19]), "=f"(r[20]), "=f"(r[21]), "=f"(r[22]),
        "=f"(r[23]), "=f"(r[24]), "=f"(r[25]), "=f"(r[26]), "=f"(r[27]), "=f"(r[28]), "=f"(r[29]),
        "=f"(r[30]), "=f"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t* r) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
      "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]),
      "r"(r[17]), "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]),
      "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
      : "memory");
}
__device__ __forceinline__ void tmem_st32f(uint32_t taddr, const float* r) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(taddr),
      "f"(r[0]), "f"(r[1]), "f"(r[2]), "f"(r[3]), "f"(r[4]), "f"(r[5]), "f"(r[6]), "f"(r[7]), "f"(r[8]),
      "f"(r[9]), "f"(r[10]), "f"(r[11]), "f"(r[12]), "f"(r[13]), "f"(r[14]), "f"(r[15]), "f"(r[16]),
      "f"(r[17]), "f"(r[18]), "f"(r[19]), "f"(r[20]), "f"(r[21]), "f"(r[22]), "f"(r[23]), "f"(r[24]),
      "f"(r[25]), "f"(r[26]), "f"(r[27]), "f"(r[28]), "f"(r[29]), "f"(r[30]), "f"(r[31])
      : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t* r) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
      "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}

// ---- descriptors ----------------------------------------------------------------------------
// Shared-memory matrix descriptor (tcgen05): start>>4 [0,14), LBO>>4 [16,30), SBO>>4 [32,46),
// version=1 [46,48), layout type [61,64) (2 = SWIZZLE_128B).
__device__ __forceinline__ uint64_t smem_desc_sw128(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= uint64_t((smem_addr & 0x3FFFF) >> 4);
  d |= uint64_t((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= uint64_t((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= uint64_t(1) << 46;
  d |= uint64_t(2) << 61;
  return d;
}
// Operand descriptor of one K = 16 step over a 2-byte tile of R sequence positions x C channels (128-byte swizzle).
// Channel-first tensors land as boxes of 64 positions ([C rows][128 B], the next 64 positions C * 128 bytes further);
// channel-last tensors as slabs of 64 channels ([R rows][128 B], the next 64 channels R * 128 bytes further) - the
// same picture with positions and channels swapped. `over_channels`: the contraction runs over the channels (Q K^T,
// dO V^T), else over the positions (P V, dS K, ...). The operand is K-major exactly when the contraction runs along
// the 128-byte rows; tile_mn_major() is the matching instruction-descriptor bit.
template <bool CL>
__host__ __device__ constexpr bool tile_mn_major(bool over_channels) {
  return CL ? !over_channels : over_channels;
}
template <bool CL>
__device__ __forceinline__ uint64_t tile_desc(uint32_t base, int ks, int R, int C, bool over_channels) {
  const uint32_t block = uint32_t(CL ? R : C) * 128u;   // bytes of one 64-wide box / slab
  if (tile_mn_major<CL>(over_channels)) return smem_desc_sw128(base + ks * 2048, block, 1024);
  return smem_desc_sw128(base + (ks >> 2) * block + (ks & 3) * 32, 16, 1024);
}
// byte offset of 8 consecutive channels [c, c + 8) of position r inside a channel-last staging tile (slabs of
// 64 channels, R rows of 128 bytes, 16-byte chunks XOR-swizzled with the row as TMA's 128-byte swizzle expects)
__device__ __forceinline__ uint32_t cl_chunk_offset(int r, int c, int R) {
  return uint32_t(c >> 6) * uint32_t(R) * 128u + uint32_t(r) * 128u + uint32_t((((c & 63) >> 3) ^ (r & 7)) << 4);
}
// MN-major 32-bit (TF32) operands must use the "128-byte swizzle with 32-byte atoms" layout (descriptor
// layout type 1; TMA swizzle CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B): the swizzle atom is 4 rows of 128 bytes.
__device__ __forceinline__ uint64_t smem_desc_sw128_base32(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= uint64_t((smem_addr & 0x3FFFF) >> 4);
  d |= uint64_t((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= uint64_t((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= uint64_t(1) << 46;
  d |= uint64_t(1) << 61;
  return d;
}
// Instruction descriptor for kind::f16 with F16 inputs and F32 accumulation.
__host__ __device__ constexpr uint32_t idesc_f16(int m, int n, bool a_mn_major, bool b_mn_major) {
  return (1u << 4)                        // c_format = F32
         | (0u << 7) | (0u << 10)         // a/b format = F16
         | (uint32_t(a_mn_major) << 15) | (uint32_t(b_mn_major) << 16) | (uint32_t(n >> 3) << 17) |
         (uint32_t(m >> 4) << 24);
}

// 16-bit element types of the tcgen05 kernels: fp16 and bf16 share every tile, descriptor and schedule; they differ in
// the a/b format bits of the kind::f16 instruction descriptor (0 = F16, 1 = BF16), the TMA data type and the float
// conversions.
template <typename T> struct Elt16;
template <> struct Elt16<__half> {
  static constexpr uint32_t kFormat = 0;
  static constexpr CUtensorMapDataType kTmaType = CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
};
template <> struct Elt16<__nv_bfloat16> {
  static constexpr uint32_t kFormat = 1;
  static constexpr CUtensorMapDataType kTmaType = CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
};
template <typename T>
__host__ __device__ constexpr uint32_t idesc_16(int m, int n, bool a_mn_major, bool b_mn_major) {
  return idesc_f16(m, n, a_mn_major, b_mn_major) | (Elt16<T>::kFormat << 7) | (Elt16<T>::kFormat << 10);
}

// Instruction descriptor for kind::tf32 (a/b format 2 = TF32) with F32 accumulation.
__host__ __device__ constexpr uint32_t idesc_tf32(int m, int n, bool a_mn_major, bool b_mn_major) {
  return (1u << 4) | (2u << 7) | (2u << 10) | (uint32_t(a_mn_major) << 15) | (uint32_t(b_mn_major) << 16) |
         (uint32_t(n >> 3) << 17) | (uint32_t(m >> 4) << 24);
}

// ---- misc -----------------------------------------------------------------------------------
template <int N>
__device__ __forceinline__ void setmaxnreg_inc() {
  asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(N));
}
template <int N>
__device__ __forceinline__ void setmaxnreg_dec() {
  asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(N));
}
__device__ __forceinline__ void named_bar_sync(uint32_t id, uint32_t nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
__device__ __forceinline__ float ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

__device__ __forceinline__ uint32_t pack_half2(float lo, float hi) {
  __half2 h = __floats2half2_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&h);
}
// two floats -> one 32-bit word of two T (round to nearest even; `lo` in the low half)
template <typename T> __device__ __forceinline__ uint32_t pack2(float lo, float hi);
template <> __device__ __forceinline__ uint32_t pack2<__half>(float lo, float hi) { return pack_half2(lo, hi); }
template <> __device__ __forceinline__ uint32_t pack2<__nv_bfloat16>(float lo, float hi) {
  uint32_t r;   // cvt packs its first source into the upper half
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}


// ---- tiles of channel-first / channel-last tensors (the CL switch of the fp16 kernels) -------------------------------
// which batch element a CTA works on: channel-first tensors index it directly, channel-last ones by (outer, head)
struct BatchCoord {
  int b, head, outer;
};
template <bool CL>
__device__ __forceinline__ BatchCoord batch_coord(int b, int heads) {
  BatchCoord c;
  c.b = b;
  c.head = CL ? b % heads : 0;
  c.outer = CL ? b / heads : b;
  return c;
}
// TMA load of a tile of R positions (a multiple of 64) x C channels (64 or 128) starting at position pos0
template <bool CL>
__device__ __forceinline__ void tile_load(uint32_t dst, const void* map, uint32_t bar, int pos0, int R, int C,
                                          const BatchCoord& bc) {
  if constexpr (CL) {
    for (int c = 0; c < C / 64; ++c) tma_load_cl(dst + c * (R * 128), map, bar, c * 64, bc.head, pos0, bc.outer);
  } else {
    for (int h = 0; h < R / 64; ++h) tma_load_bc(dst + h * (C * 128), map, bar, pos0 + h * 64, bc.b);
  }
}
// TMA store of a staged tile (stage_row32 layout); n = the tensor's sequence length
template <bool CL>
__device__ __forceinline__ void tile_store(const void* map, uint32_t src, int pos0, int R, int C, int n,
                                           const BatchCoord& bc) {
  if constexpr (CL) {
    for (int c = 0; c < C / 64; ++c) tma_store_cl(map, src + c * (R * 128), c * 64, bc.head, pos0, bc.outer);
  } else {
    for (int h = 0; h < R / 64; ++h)
      if (pos0 + h * 64 < n) tma_store_bc(map, src + h * (C * 128), pos0 + h * 64, bc.b);
  }
}
// One thread owns row r of an output tile and stages channels [c0, c0 + 32) = v[0..32) * scale as T.
// channel-first: [C][64] per 64 positions, unswizzled (lanes = consecutive positions: conflict-free 2-byte stores);
// channel-last: slabs of 64 channels, rows of 128 bytes with TMA's 128-byte swizzle (16-byte stores, conflict-free)
template <bool CL, typename T>
__device__ __forceinline__ void stage_row32(uint8_t* tile, int r, int c0, int R, int C, const float* v, float scale) {
  if constexpr (CL) {
#pragma unroll
    for (int e = 0; e < 32; e += 8) {
      uint4 w;
      w.x = pack2<T>(v[e] * scale, v[e + 1] * scale);
      w.y = pack2<T>(v[e + 2] * scale, v[e + 3] * scale);
      w.z = pack2<T>(v[e + 4] * scale, v[e + 5] * scale);
      w.w = pack2<T>(v[e + 6] * scale, v[e + 7] * scale);
      *reinterpret_cast<uint4*>(tile + cl_chunk_offset(r, c0 + e, R)) = w;
    }
  } else {
    T* h = reinterpret_cast<T*>(tile) + (r >> 6) * (C * 64) + (r & 63);
#pragma unroll
    for (int e = 0; e < 32; ++e) h[(c0 + e) * 64] = from_acc<T>(v[e] * scale);
  }
}
// zeros are the same bits in fp16 and bf16: one version serves both
template <bool CL>
__device__ __forceinline__ void stage_row_zero(uint8_t* tile, int r, int c_begin, int c_end, int R, int C) {
  if constexpr (CL) {
    for (int c = c_begin; c < c_end; c += 8)
      *reinterpret_cast<uint4*>(tile + cl_chunk_offset(r, c, R)) = make_uint4(0, 0, 0, 0);
  } else {
    __half* h = reinterpret_cast<__half*>(tile) + (r >> 6) * (C * 64) + (r & 63);
    for (int c = c_begin; c < c_end; ++c) h[c * 64] = __float2half_rn(0.f);
  }
}

}  // namespace ptx
}  // namespace fa
