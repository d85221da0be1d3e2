// PTX wrappers shared by the tcgen05 kernels (gemm_tcgen05.cu, attn_tc.cu): mbarriers, TMA tensor loads, tcgen05
// fences / commits / MMA, UMMA shared-memory descriptors, and the host-side tensor-map encoder.
#pragma once
#include <cuda.h>

#include "common.cuh"

namespace ltm {

// Host: 2-D fp32 tensor map {inner, outer} with row pitch `pitch_elems`, box {box_inner, box_outer};
// swizzle32b_atom = 0: SWIZZLE_128B (K-major operands), 1: SWIZZLE_128B_ATOM_32B (MN-major fp32 operands).
int tma_encode_2d(CUtensorMap* map, const float* base, unsigned long long inner, unsigned long long outer,
                  unsigned long long pitch_elems, unsigned box_inner, unsigned box_outer, int swizzle32b_atom,
                  const char* what);
// Host: 2-D fp16 tensor map {inner halves, outer rows} with row pitch `pitch_elems` halves, box {64, box_outer},
// SWIZZLE_128B.
int tma_encode_2d_f16(CUtensorMap* map, const void* base, unsigned long long inner, unsigned long long outer,
                      unsigned long long pitch_elems, unsigned box_outer, const char* what);

#ifdef __CUDACC__
// ------------------------------------------------------------------------------------------ PTX
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ uint32_t mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t done;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(done)
      : "r"(bar), "r"(parity)
      : "memory");
  return done;
}
// Bounded wait: a broken pipeline traps (launch error) after ~2 s instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  unsigned long long t0;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if ((++spins & 0x3fffu) == 0) {
      unsigned long long t1;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
      if (t1 - t0 > 2000000000ull) {
        printf("libinfltm gemm: mbarrier wait timed out (block %d,%d,%d thread %d)\n", blockIdx.x, blockIdx.y,
               blockIdx.z, threadIdx.x);
        asm volatile("trap;");
      }
    }
  }
}
__device__ __forceinline__ void tma_load_3d(const CUtensorMap* map, uint32_t dst, uint32_t bar, int c0, int c1,
                                            int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tcgen05_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tcgen05_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tcgen05_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// The descriptors are passed as (low word, high word): only the low word (start address | LBO) changes from MMA
// to MMA, by a constant step, so the issuing thread spends one add per operand instead of rebuilding 64-bit
// descriptors (the first version's ~40 instructions per MMA on a single thread cost more than the MMA's 128 cycles).
__device__ __forceinline__ void tcgen05_mma_tf32(uint32_t tmem_d, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo,
                                                 uint32_t b_hi, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
      "setp.ne.b32 p, %6, 0;\n\t"
      "mov.b64 da, {%1, %2};\n\t"
      "mov.b64 db, {%3, %4};\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], da, db, %5, p;\n\t}"
      ::"r"(tmem_d), "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate)
      : "memory");
}

// UMMA shared-memory matrix descriptor (sm_100): start>>4 [0,14) | LBO>>4 [16,30) | SBO>>4 [32,46) |
// version=1 [46,48) | layout type [61,64): SWIZZLE_128B = 2, SWIZZLE_128B_BASE32B = 1.
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes,
                                              uint32_t layout) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32;
  d |= 1ull << 46;
  d |= (uint64_t)layout << 61;
  return d;
}
// fp16 operands (kind::f16, K = 16 per instruction), fp32 accumulate
__device__ __forceinline__ void tcgen05_mma_f16(uint32_t tmem_d, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo,
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
__device__ __forceinline__ void tma_load_2d(const CUtensorMap* map, uint32_t dst, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ float tf32_rna(float x) {       // round to nearest (ties away) onto the tf32 grid
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return __uint_as_float(r);
}
#endif

}  // namespace ltm
