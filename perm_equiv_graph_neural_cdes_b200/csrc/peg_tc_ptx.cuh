// Hand-written PTX wrappers shared by the tcgen05 kernels (peg_tc.cu: 3xTF32 operands; peg_tc16.cu: bf16x2 operands).
#pragma once
#include <cuda.h>
#include <stdint.h>

namespace peg {

// ------------------------------------------------------------------------------------------
// PTX wrappers
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.shared::cta.b64 st, [%0];\n\t}" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.expect_tx.shared::cta.b64 st, [%0], %1;\n\t}" ::"r"(bar), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra DONE_%=;\n\t"
      "bra WAIT_%=;\n\t"
      "DONE_%=:\n\t"
      "}" ::"r"(bar),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(dst),
      "l"(map), "r"(c0), "r"(c1), "r"(bar)
      : "memory");
}

__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accum)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// streaming 128-bit plane loads.  Measured on B200 (n=2048, d=128, B=9, forward launch): ld.global.cg 137.6 us, ld.global.nc 139.6,
// ld.global.nc.L1::no_allocate 156.1, ld.global.cs 159.8, ...no_allocate.L2::256B 156.7 -- the adjoint is insensitive (217 us)
__device__ __forceinline__ float4 ldg_stream(const float* p) {
  float4 r;
  asm volatile("ld.global.cg.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
  return r;
}

__device__ __forceinline__ float tf32_rna(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return __uint_as_float(r);
}

// K-major SWIZZLE_128B shared-memory matrix descriptor (rows of 128 B, 8-row groups 1024 B apart)
__device__ __forceinline__ uint64_t make_desc_sw128(uint32_t saddr) {
  return (uint64_t)((saddr >> 4) & 0x3FFF) | (1ull << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}


// K-major SWIZZLE_64B shared-memory matrix descriptor (rows of 64 B = 32 bf16, 8-row groups 512 B apart)
__device__ __forceinline__ uint64_t make_desc_sw64(uint32_t saddr) {
  return (uint64_t)((saddr >> 4) & 0x3FFF) | (1ull << 16) | (32ull << 32) | (1ull << 46) | (4ull << 61);
}

__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accum)
      : "memory");
}

// two fp32 -> packed bf16x2 (round to nearest even); `lo` lands in the low half = the lower address
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
// bf16x2 split of two fp32 values: x = hi + lo + O(2^-17 |x|); both parts packed like pack_bf16x2
__device__ __forceinline__ void split_bf16x2(float x0, float x1, uint32_t& hi, uint32_t& lo) {
  hi = pack_bf16x2(x0, x1);
  const float r0 = x0 - __uint_as_float(hi << 16);
  const float r1 = x1 - __uint_as_float(hi & 0xffff0000u);
  lo = pack_bf16x2(r0, r1);
}

// fp16x2 split of two fp32 values (already scaled into the fp16 range): x = hi + lo + O(2^-22 |x|).
// hi = x rounded to 11 significant bits IN the fp32 word (add half an ulp of the 11-bit grid to the bit pattern, clear the 13 low
// mantissa bits: round-half-away, symmetric about zero; two integer instructions -- cvt.rna.tf32.f32 would do the same but ptxas
// expands it to four with its NaN handling), so hi is exactly representable in fp16 and the residual lo = x - hi needs no
// fp16 -> fp32 conversion.  The rounding must be symmetric: with truncation lo always has the sign of x, the dropped lo*lo product
// becomes a systematic bias and the param1/param2 gradients (sums with ~1e3-fold cancellation) lose their 3e-4 parity (measured).
// Below the fp16 normal range (|x| < 2^-14 after scaling = 2^-28 of the block maximum) the pack rounds hi once more: <= 2^-25 absolute.
__device__ __forceinline__ void split_f16x2(float x0, float x1, uint32_t& hi, uint32_t& lo) {
  const float h0 = __uint_as_float((__float_as_uint(x0) + 0x1000u) & 0xffffe000u), h1 = __uint_as_float((__float_as_uint(x1) + 0x1000u) & 0xffffe000u);
  asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(hi) : "f"(h1), "f"(h0));
  asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(lo) : "f"(x1 - h1), "f"(x0 - h0));
}

}  // namespace peg
