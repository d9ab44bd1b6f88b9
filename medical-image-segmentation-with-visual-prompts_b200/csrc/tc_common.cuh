// Thin inline-PTX layer over the Blackwell (sm_100a) tensor-core path: tcgen05.mma with TMEM accumulators,
// TMEM alloc/ld/st, mbarrier, proxy fences, and shared-memory matrix descriptors (no-swizzle canonical layouts).
// Bit layouts follow the PTX ISA "tcgen05" chapter (cross-checked against cute/arch/mma_sm100_desc.hpp).
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <stdio.h>

namespace pwa {
namespace tc {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ---- mbarrier ----------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
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
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
#ifdef PWA_WATCHDOG   // debug builds (make WATCHDOG=1): report a wait that never completes instead of hanging the GPU
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++spins > (1u << 24)) {
      printf("pwa watchdog: block %d thread %d stuck on mbarrier smem 0x%x parity %u\n", (int)blockIdx.x, (int)threadIdx.x,
             smem_u32(bar), parity);
      __trap();
    }
  }
#else
  while (!mbar_try_wait(bar, parity)) {
  }
#endif
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// one lane of the (converged) warp; lets ptxas keep warp-uniform operands of the guarded instructions in uniform registers
__device__ __forceinline__ bool elect_one_sync() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}

// transaction bytes the current phase of the barrier additionally waits for (bulk copies complete them)
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.expect_tx.relaxed.cta.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// contiguous global -> shared bulk copy (16-byte aligned, size a multiple of 16), completion counted on `bar`
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst_smem)),
               "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// generic-proxy smem writes (st.shared) -> visible to the async proxy (tcgen05.mma operand reads)
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ---- TMEM --------------------------------------------------------------------------------------
// Whole-warp, .sync.aligned.  ncols: power of two in [32, 512].  Writes the base address to *dst_smem.
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// TMEM address = (lane << 16) | column.  A warp may only touch lanes [32*(warp%4), +32).
// 32x32b.x32: thread t of the warp receives lane (base_lane + t), columns [col, col+32).
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
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
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
      "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}

__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t (&r)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(r[0]), "r"(r[1]),
               "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
               : "memory");
}

// ---- descriptors -------------------------------------------------------------------------------
// Shared-memory matrix descriptor, SWIZZLE_NONE.  All byte quantities are multiples of 16.
//   K-major  operand [rows][K]: element (r,k) at (r%8)*16 + (r/8)*SBO + (k/8)*LBO + (k%8)*2
//   MN-major operand [K][mn]  : element (k,m) at (m%8)*2  + (k%8)*16  + (m/8)*SBO + (k/8)*LBO
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= 1ull << 46;  // descriptor version (Blackwell)
  return d;         // base_offset = 0, lbo_mode = 0, layout_type = SWIZZLE_NONE (0)
}

// A / B format code of a kind::f16 instruction descriptor (bits 7-9 and 10-12): F16 = 0, BF16 = 1
template <typename T> struct F16Kind;
template <> struct F16Kind<__nv_bfloat16> { static constexpr uint32_t fmt = 1; };
template <> struct F16Kind<__half> { static constexpr uint32_t fmt = 0; };

// Instruction descriptor for kind::f16, T x T -> fp32 (T = bf16 or fp16), dense.
template <typename T>
__host__ __device__ constexpr uint32_t make_idesc(int M, int N, int a_mn_major, int b_mn_major) {
  return (1u << 4) | (F16Kind<T>::fmt << 7) | (F16Kind<T>::fmt << 10) | ((uint32_t)a_mn_major << 15) | ((uint32_t)b_mn_major << 16) |
         ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__host__ __device__ constexpr uint32_t make_idesc_bf16(int M, int N, int a_mn_major, int b_mn_major) {
  return make_idesc<__nv_bfloat16>(M, N, a_mn_major, b_mn_major);
}

// D[tmem] (+)= A[smem] * B[smem]      (single thread issues)
__device__ __forceinline__ void mma_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accum)
      : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem]
__device__ __forceinline__ void mma_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}" ::"r"(d_tmem),
      "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accum)
      : "memory");
}
// all previously issued MMAs of this thread -> arrive(1) on the mbarrier when complete
__device__ __forceinline__ void mma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}

__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);  // .x = lo (low 16 bits)
  return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ uint32_t pack_f16(float lo, float hi) {
  __half2 v = __floats2half2_rn(lo, hi);             // .x = lo (low 16 bits); overflow rounds to +-inf, NaN stays NaN
  return *reinterpret_cast<uint32_t*>(&v);
}
// pair pack / unpack of the element type T (bf16 or fp16) of the tcgen05 kernels
template <typename T> __device__ __forceinline__ uint32_t pack2t(float lo, float hi);
template <> __device__ __forceinline__ uint32_t pack2t<__nv_bfloat16>(float lo, float hi) { return pack_bf16(lo, hi); }
template <> __device__ __forceinline__ uint32_t pack2t<__half>(float lo, float hi) { return pack_f16(lo, hi); }
template <typename T> __device__ __forceinline__ void unpack2t(uint32_t w, float& lo, float& hi);
template <> __device__ __forceinline__ void unpack2t<__nv_bfloat16>(uint32_t w, float& lo, float& hi) {
  lo = __uint_as_float(w << 16);
  hi = __uint_as_float(w & 0xffff0000u);
}
template <> __device__ __forceinline__ void unpack2t<__half>(uint32_t w, float& lo, float& hi) {
  const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&w));
  lo = f.x;
  hi = f.y;
}

}  // namespace tc
}  // namespace pwa
