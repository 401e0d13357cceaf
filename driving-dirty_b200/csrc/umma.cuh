// Minimal sm_100a tcgen05 / TMEM / mbarrier / TMA wrappers (inline PTX) shared by every tensor-core kernel of the
// library (conv_tc.cu, conv_wgrad_tc.cu, conv_dil_tc.cu, conv_dil_wgrad_tc.cu, linear_tc.cu) and the probes in tools/.
// This is the only place that waits on an mbarrier.  Descriptor bit layouts follow the PTX ISA "matrix descriptor" /
// "instruction descriptor" tables (same fields as cute::UMMA::SmemDescriptor / InstrDescriptor).
#pragma once
#include <cuda_bf16.h>
#include <stdint.h>

namespace umma {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// true in exactly one (converged) lane of the warp; keeps the surrounding code warp-uniform so that
// descriptors / addresses can live in uniform registers (a lone divergent thread pays an R2UR chain
// of ~145 cycles per tcgen05.mma -- measured with tools/umma_rate.cu)
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}

// ---------------------------------------------------------------- mbarrier ----------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// arrival without release semantics: a default (.release) arrive first drains the warp's outstanding global
// stores (~700 cycles per epilogue row measured in conv3x3_c32_s1_tc_kernel).  For hand-offs whose only payload
// is "my tcgen05.ld has completed" (tcgen05.wait::ld + tcgen05.fence::before_thread_sync order that).
__device__ __forceinline__ void mbar_arrive_relaxed(uint64_t* bar) {
  asm volatile("mbarrier.arrive.relaxed.cta.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: a protocol bug traps (reported as a launch failure) instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++spins > (1u << 22)) __trap();
  }
}
// The same bound, backing off between polls: for waiters (epilogue and store warps) that would otherwise take issue
// slots from the producer / MMA warps sharing their schedulers.
__device__ __forceinline__ void mbar_wait_sleep(uint64_t* bar, uint32_t parity) {
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    __nanosleep(64);
    if (++spins > (1u << 22)) __trap();
  }
}

// ---------------------------------------------------------------- proxies / fences --------
// generic-proxy smem writes (st.shared, cp.async) -> visible to the async proxy (UMMA, TMA)
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_before_sync() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after_sync() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}

// ---------------------------------------------------------------- TMEM --------------------
// whole warp; writes the allocated base address to *dst (shared memory)
__device__ __forceinline__ void tmem_alloc(uint32_t* dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst)), "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// whole CTA, after one warp's tmem_alloc(slot, ...): returns the allocated base to every thread
__device__ __forceinline__ uint32_t tmem_publish(uint32_t* slot) {
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  return __shfl_sync(0xffffffffu, *slot, 0);
}

// 32 lanes x 32 columns of fp32: thread i of the warp gets lane (base_lane + i), columns c..c+31
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
// 32 lanes x 16 columns of fp32
__device__ __forceinline__ void tmem_ld_32x16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
// 32 lanes x 4 columns of fp32
__device__ __forceinline__ void tmem_ld_32x4(uint32_t taddr, uint32_t (&r)[4]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(taddr)
               : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ---------------------------------------------------------------- descriptors -------------
// shared-memory matrix descriptor, SWIZZLE_NONE ("interleave": 8x16B core matrices, 128 B each)
//   K-major : 8 MN-rows x 16 B per core matrix; LBO = byte stride between the K core matrices,
//             SBO = byte stride between 8-row groups along M/N
//   MN-major: 8 K-rows x 16 B (8 MN elements) per core matrix; SBO = stride between 8-element MN
//             chunks, LBO = stride between 8-row K groups
__device__ __forceinline__ uint64_t make_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;   // descriptor version (Blackwell)
  return d;                 // base_offset 0, lbo_mode 0, layout_type 0 = SWIZZLE_NONE
}

// Split form for hot issue loops: the high word is constant per operand kind, the low word is
// (start address >> 4) | (LBO >> 4) << 16, so advancing an operand is ONE 32-bit add.
__device__ __forceinline__ uint32_t desc_lo(uint32_t smem_addr, uint32_t lbo_bytes) {
  return ((smem_addr >> 4) & 0x3FFF) | (((lbo_bytes >> 4) & 0x3FFF) << 16);
}
__host__ __device__ constexpr uint32_t desc_hi(uint32_t sbo_bytes) {
  return ((sbo_bytes >> 4) & 0x3FFF) | (1u << 14);   // version bit 46 -> bit 14 of the high word
}

// kind::f16 instruction descriptor: bf16 x bf16 -> fp32
__host__ __device__ constexpr uint32_t make_idesc_bf16(int M, int N, bool a_mn_major, bool b_mn_major) {
  return (1u << 4)                       // c_format = F32
         | (1u << 7)                     // a_format = BF16
         | (1u << 10)                    // b_format = BF16
         | ((a_mn_major ? 1u : 0u) << 15)
         | ((b_mn_major ? 1u : 0u) << 16)
         | ((uint32_t)(N >> 3) << 17)
         | ((uint32_t)(M >> 4) << 24);
}

// D[tmem] (+)= A[smem] * B[smem]; issued by ONE thread
__device__ __forceinline__ void mma_bf16(uint32_t tmem_d, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                         uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void mma_bf16_lohi(uint32_t tmem_d, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo,
                                              uint32_t b_hi, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
      "setp.ne.b32 p, %6, 0;\n\t"
      "mov.b64 da, {%1, %2};\n\t"
      "mov.b64 db, {%3, %4};\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, p;\n\t}"
      ::"r"(tmem_d), "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrive on an mbarrier when all tcgen05.mma issued so far by this thread have completed
__device__ __forceinline__ void mma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}

// ---------------------------------------------------------------- 256-bit global access ---
// sm_100 32-byte vector load / store (pointer 32-byte aligned): one whole sector per lane
__device__ __forceinline__ void ldg256(const void* p, uint32_t* v) {
  asm volatile("ld.global.nc.v8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
               : "l"(p));
}
__device__ __forceinline__ void stg256(void* p, const uint32_t* v) {
  asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(p), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]),
               "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7])
               : "memory");
}

}  // namespace umma

// ---------------------------------------------------------------- 128B-swizzled operands / TMA ----
namespace umma {

// shared-memory matrix descriptor, SWIZZLE_128B (what a TMA box with a 128-byte inner extent and
// CU_TENSOR_MAP_SWIZZLE_128B produces; tile base 1024-byte aligned):
//   K-major : rows of 128 B (one swizzle span of K), 8-row atoms of 1024 B; SBO = stride between 8-row
//             groups along M/N; LBO unused; advancing K inside the span = start address + bytes
//   MN-major: rows = K index, 128 B = 32 fp32 (64 bf16) MN elements; LBO = stride between MN blocks,
//             SBO = stride between groups of 8 K rows
__device__ __forceinline__ uint32_t desc_hi_sw128(uint32_t sbo_bytes) {
  return ((sbo_bytes >> 4) & 0x3FFF) | (1u << 14) | (2u << 29);   // version 1, layout_type 2 = SWIZZLE_128B (bits 61-63)
}
// SWIZZLE_64B (layout_type 4): what a whole-pixel TMA box of a 32-channel bf16 NHWC row produces (64-byte rows, 8-row atoms of
// 512 B).  K-major: rows = M/N index, SBO = stride between 8-row groups, K advances inside the row (+32 B per K = 16).
// MN-major: rows = K index, LBO = stride between 32-element MN blocks, SBO = stride between 8-row K groups.
// The swizzle follows the absolute shared-memory address: a start address shifted by whole rows works with base_offset 0.
__host__ __device__ constexpr uint32_t desc_hi_sw64(uint32_t sbo_bytes) {
  return ((sbo_bytes >> 4) & 0x3FFF) | (1u << 14) | (4u << 29);
}
// SWIZZLE_128B_BASE32B (layout_type 1): the only layout for MN-major tf32 operands; 4-row K atoms
// (TMA: CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B); SBO = stride between groups of 4 K rows
__device__ __forceinline__ uint32_t desc_hi_sw128_base32(uint32_t sbo_bytes) {
  return ((sbo_bytes >> 4) & 0x3FFF) | (1u << 14) | (1u << 29);
}

// kind::tf32 instruction descriptor: tf32 x tf32 -> fp32 (operands are fp32 words in shared memory)
__host__ __device__ constexpr uint32_t make_idesc_tf32(int M, int N, bool a_mn_major, bool b_mn_major) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((a_mn_major ? 1u : 0u) << 15) | ((b_mn_major ? 1u : 0u) << 16) |
         ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ void mma_tf32_lohi(uint32_t tmem_d, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi,
                                              uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
      "setp.ne.b32 p, %6, 0;\n\t"
      "mov.b64 da, {%1, %2};\n\t"
      "mov.b64 db, {%3, %4};\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], da, db, %5, p;\n\t}"
      ::"r"(tmem_d), "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate)
      : "memory");
}

// TMA: 2-D tile global -> shared, completion counted in bytes on an mbarrier.  c0 = innermost coordinate.
__device__ __forceinline__ void tma_load_2d(uint32_t dst_smem, const void* tmap, int c0, int c1, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst_smem), "l"(tmap), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
// 4-D tile (c0 = innermost coordinate); out-of-range elements are written as zeros and count towards the transaction bytes
__device__ __forceinline__ void tma_load_4d(uint32_t dst_smem, const void* tmap, int c0, int c1, int c2, int c3, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(dst_smem), "l"(tmap), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const void* tmap) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(tmap) : "memory");
}
// TMA: 2-D tile shared -> global (out-of-range elements are not written).  The writers of the tile must have run
// fence_proxy_async_smem() and synchronised with the issuing thread first.
__device__ __forceinline__ void tma_store_2d(const void* tmap, uint32_t src_smem, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
               ::"l"(tmap), "r"(src_smem), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void bulk_commit_group() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// at most N committed bulk groups of this thread still READ their shared-memory source (the source may then be reused)
template <int N>
__device__ __forceinline__ void bulk_wait_group_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
// at most N committed bulk groups of this thread are still incomplete (writes visible in global memory)
template <int N>
__device__ __forceinline__ void bulk_wait_group() {
  asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}

}  // namespace umma
