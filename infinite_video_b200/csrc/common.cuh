// Shared helpers for the libinfltm kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/infltm.h"

namespace ltm {

void set_error(const char* fmt, ...);

#define LTM_REQUIRE(cond, ...)                  \
  do {                                          \
    if (!(cond)) {                              \
      ::ltm::set_error(__VA_ARGS__);            \
      return -1;                                \
    }                                           \
  } while (0)

#define LTM_CHECK_LAUNCH(name)                                                        \
  do {                                                                                \
    cudaError_t _e = cudaGetLastError();                                              \
    if (_e != cudaSuccess) {                                                          \
      ::ltm::set_error("%s: launch failed: %s", name, cudaGetErrorString(_e));        \
      return -2;                                                                      \
    }                                                                                 \
  } while (0)

#define LTM_CUDA(call)                                                                \
  do {                                                                                \
    cudaError_t _e = (call);                                                          \
    if (_e != cudaSuccess) {                                                          \
      ::ltm::set_error("%s failed: %s", #call, cudaGetErrorString(_e));               \
      return -3;                                                                      \
    }                                                                                 \
  } while (0)

static inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// Frame pooling behind every ltm_pool_* entry point and the step: checks the arguments (`who` names the caller in the
// error text), picks the kernel, thread count and grid.  k[Bv, L, T, e], dtype 0 fp32, 1 fp16, 2 bfloat16, is pooled
// into xpart as the frame means in `splits` partial sums, [Bv*L, splits, e]; offs != NULL: only the `frames` frames of
// a ragged chunk (ltm_pool_mean_ragged), packed; fbin_ptr != NULL: the per-bin sums [Bv, rows, e] instead
// (ltm_pool_bins); k16 != NULL: the chunk as fp16 as well (ltm_pool_mean_convert, ld16 rows per video when ragged);
// ptrs != NULL (with offs, k == NULL): the ragged chunk of video v read from ptrs[v] instead of k[v]
// (ltm_pool_mean_ptrs).  max_ctas > 0 bounds the grid of the per-frame means (0 = one CTA per (frame, token-split)).
int pool_frames(const char* who, const void* k, int dtype, float* xpart, int Bv, int L, int T, int e, int splits,
                int max_ctas, void* stream, const int32_t* offs = nullptr, int frames = 0, void* k16 = nullptr,
                int ld16 = 0, const int32_t* fbin_ptr = nullptr, int rows = 0, const void* const* ptrs = nullptr);

// ---- ragged batches (ltm_rect_step_args.lengths), internal to the library
// ltm_consolidate_rect_kv with per-video lengths (0 = idle) and frame offsets; NULL lengths = lock-step
int consolidate_rect_ragged(const float* B_past, const float* xpart, const int32_t* idx, int64_t idx_stride,
                            const uint8_t* new_doc, const int32_t* seg_ptr0, const int32_t* seg_mem0, const float* g0,
                            const int32_t* seg_ptr1, const int32_t* seg_mem1, const float* g1, float* B_new,
                            void* B_half, const float* KV_past, float* KV_new, const float* bkv, int ldkv, int jf,
                            int round_tf32, int Bv, int N, int e, int L, int splits, int S, const int32_t* lengths,
                            const int32_t* offs, void* stream);
// dst[v] = src[v] (src NULL: zeros) over bytes_per_video for the videos with lengths[v] == 0
int carry_idle(const int32_t* lengths, const void* src, void* dst, size_t bytes_per_video, int Bv, void* stream);
// ltm_resample that skips (reads no uniforms of, writes nothing for) the videos with lengths[v] == 0
int resample_ragged(const float* hist_part, int parts, int ncat, int normalize, const double* u, const float* bins,
                    const int32_t* bin2basis, int sort, float* p_out, int32_t* b_draw, int32_t* b_used, float* ts,
                    int32_t* idx, int Bv, int S, const int32_t* lengths, void* stream);

// The dynamic-shared-memory opt-in of a kernel and the SM count are properties of a DEVICE, so their one-time setup
// is cached per device ordinal (a process may drive several GPUs: a Q-former sharded with device_map).
constexpr int LTM_MAX_DEVICES = 64;
struct PerDevice {
  size_t smem[LTM_MAX_DEVICES];      // largest dynamic shared memory size opted into so far
  int num_sms[LTM_MAX_DEVICES];
};
template <class Kern>
static inline int kernel_setup(Kern kern, size_t smem_bytes, PerDevice& pd, int* num_sms) {
  int dev = 0;
  LTM_CUDA(cudaGetDevice(&dev));
  LTM_REQUIRE(dev >= 0 && dev < LTM_MAX_DEVICES, "device ordinal %d out of range", dev);
  if (smem_bytes > pd.smem[dev]) {
    LTM_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes));
    pd.smem[dev] = smem_bytes;
  }
  if (pd.num_sms[dev] == 0)
    LTM_CUDA(cudaDeviceGetAttribute(&pd.num_sms[dev], cudaDevAttrMultiProcessorCount, dev));
  if (num_sms) *num_sms = pd.num_sms[dev];
  return 0;
}

#ifdef __CUDACC__
// 128-bit streaming load: read-only path, no L1 allocation, L2 evict-first (data is touched once).
__device__ __forceinline__ float4 ldg_stream(const float4* p, uint64_t policy) {
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.f32 {%0,%1,%2,%3}, [%4], %5;"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
               : "l"(p), "l"(policy));
  return r;
}
__device__ __forceinline__ uint64_t policy_evict_first() {
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ uint64_t policy_evict_last() {
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ float4 ldg_nc(const float4* p) {
  float4 r;
  asm volatile("ld.global.nc.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
               : "l"(p));
  return r;
}
__device__ __forceinline__ void f4_add(float4& a, const float4& b) {
  a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w;
}
// the same four IEEE additions as two packed instructions (sm_100 add.rn.f32x2): half the issue slots of the
// accumulation in the streaming kernels
__device__ __forceinline__ void f4_add_packed(float4& a, const float4& b) {
  unsigned long long a0, a1, b0, b1;
  asm("mov.b64 %0, {%1, %2};" : "=l"(a0) : "f"(a.x), "f"(a.y));
  asm("mov.b64 %0, {%1, %2};" : "=l"(a1) : "f"(a.z), "f"(a.w));
  asm("mov.b64 %0, {%1, %2};" : "=l"(b0) : "f"(b.x), "f"(b.y));
  asm("mov.b64 %0, {%1, %2};" : "=l"(b1) : "f"(b.z), "f"(b.w));
  asm("add.rn.f32x2 %0, %0, %1;" : "+l"(a0) : "l"(b0));
  asm("add.rn.f32x2 %0, %0, %1;" : "+l"(a1) : "l"(b1));
  asm("mov.b64 {%0, %1}, %2;" : "=f"(a.x), "=f"(a.y) : "l"(a0));
  asm("mov.b64 {%0, %1}, %2;" : "=f"(a.z), "=f"(a.w) : "l"(a1));
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
#endif

}  // namespace ltm
