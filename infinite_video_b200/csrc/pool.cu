// R4 -- frame pooling: x[v,l,:] = mean_t k[v,l,t,:]   (long_term_attention_gibbs.py:304; the
// VideoChat2 copy pools 14x14 tokens of width 1024, VCB/long_term_attention_gibbs.py:304).
//
// This kernel moves >90 % of the algorithmic bytes of a variant-R call (L*T*e*4 of the
// 4*(L*T*e + 2*Q*D + 2*N*e) + 8*S bytes), so it is a pure HBM streamer: one CTA per
// (frame, token-split), one thread per 128-bit column group, 8 independent 128-bit loads in
// flight per thread through the read-only path with no L1 allocation and an L2 evict-first
// policy (the chunk is read exactly once).  Partial sums over `splits` token ranges are kept
// separate (deterministic, no atomics) and added by the consolidation kernel; splits > 1 only
// exists to fill the 148 SMs when Bv*L is small.
#include <cuda_fp16.h>

#include "common.cuh"

namespace ltm {

constexpr int POOL_UNROLL = 8;
constexpr int POOL_ACC = 2;

// Sum of the token rows [r0, r1) of one frame for the 128-bit column group c: 8 independent 128-bit loads in flight,
// folded into two accumulators (the register file is what limits how many of these CTAs fit next to the
// compute-bound kernels of the other stream: 44 registers -> 7 per SM).  Every pooling kernel goes through this
// function, so the summation order -- and with it every bit of the pooled frame -- is the same in all of them.
__device__ __forceinline__ float4 pool_rows(const float4* __restrict__ base, int r0, int r1, int e4, int c,
                                            uint64_t pol) {
  float4 acc[POOL_ACC];
#pragma unroll
  for (int i = 0; i < POOL_ACC; ++i) acc[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  int r = r0;
  for (; r + POOL_UNROLL <= r1; r += POOL_UNROLL) {
    float4 v[POOL_UNROLL];
#pragma unroll
    for (int i = 0; i < POOL_UNROLL; ++i) v[i] = ldg_stream(base + (size_t)(r + i) * e4 + c, pol);
#pragma unroll
    for (int i = 0; i < POOL_UNROLL; ++i) f4_add_packed(acc[i % POOL_ACC], v[i]);
  }
  for (; r < r1; ++r) f4_add(acc[0], ldg_stream(base + (size_t)r * e4 + c, pol));
#pragma unroll
  for (int i = 1; i < POOL_ACC; ++i) f4_add(acc[0], acc[i]);
  return acc[0];
}

// Token-split `sp` of frame `src` of the chunk, written to row (unit * splits + sp) of xpart: the threads of the CTA
// each own 128-bit column groups.
__device__ __forceinline__ void pool_unit_at(const float4* __restrict__ k, float4* __restrict__ xpart, int T, int e4,
                                             int splits, float Tf, unsigned unit, int sp, size_t src, uint64_t pol) {
  const int r0 = (int)(((long long)T * sp) / splits);
  const int r1 = (int)(((long long)T * (sp + 1)) / splits);
  const float4* base = k + src * T * e4;
  for (int c = threadIdx.x; c < e4; c += blockDim.x) {
    float4 o = pool_rows(base, r0, r1, e4, c, pol);
    // torch.mean == sum / T (true division, so T = 196 rounds like the reference).  With splits > 1 (small batches
    // only) every partial sum is divided -- and rounded -- on its own and the consumer adds the partial means: the
    // pooled frame then differs from sum / T by up to `splits` ulp (1e-7 relative; the coefficient tolerance is 1e-5).
    o.x = __fdiv_rn(o.x, Tf); o.y = __fdiv_rn(o.y, Tf); o.z = __fdiv_rn(o.z, Tf); o.w = __fdiv_rn(o.w, Tf);
    xpart[((size_t)unit * splits + sp) * e4 + c] = o;
  }
}

// One (frame, token-split) work item of a lock-step chunk: frame unit = v*L + l in and out.
__device__ __forceinline__ void pool_unit(const float4* __restrict__ k, float4* __restrict__ xpart, int T, int e4,
                                          int splits, float Tf, unsigned work, uint64_t pol) {
  const unsigned unit = work / splits;
  pool_unit_at(k, xpart, T, e4, splits, Tf, unit, (int)(work - unit * splits), unit, pol);
}

// Frame pooling folded with the first half of the regression (VERDICT r1, "bin sums instead of xpart"): the frames of
// an update chunk that fall into the same basis bin are consecutive (tables.py: fbin_ptr), and the consolidation only
// ever needs their sum, so one CTA per (video, bin) pools its frames one after the other -- each exactly like
// pool_unit with splits == 1 -- and writes the running sum of the frame means: xbin[v, r, :] = sum_f mean_t k[v,f,t,:].
// At the NExT-QA shape that is 64 rows per video instead of 256 (0.2 instead of 0.8 MB written and read back).
// (Measured alternatives: FP = 2..4 frames of a bin side by side in one CTA of FP x 192 threads, frame means staged in
// shared memory.  Alone on the GPU that is the fastest pooling kernel of all -- 0.4645 ms for 3.2 GB at FP = 4 -- but
// next to the other stream's kernels its large CTAs lose: 188.6 k chunks/s at FP = 4, 192.9 k at FP = 2, against
// 194.4 k for this one-frame-at-a-time form, whose CTAs hold 7.7 k registers each and leave room sooner.)
__global__ void __launch_bounds__(256)
pool_bins_kernel(const float4* __restrict__ k, float4* __restrict__ xbin, const int32_t* __restrict__ fbin_ptr,
                 int L, int T, int e4, int rows, float Tf) {
  const uint64_t pol = policy_evict_first();
  const int r = blockIdx.x, v = blockIdx.y;
  const int f0 = fbin_ptr[r], f1 = fbin_ptr[r + 1];
  const float4* kv = k + (size_t)v * L * T * e4;
  for (int c = threadIdx.x; c < e4; c += blockDim.x) {
    float4 sum = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int f = f0; f < f1; ++f) {
      float4 o = pool_rows(kv + (size_t)f * T * e4, 0, T, e4, c, pol);
      o.x = __fdiv_rn(o.x, Tf); o.y = __fdiv_rn(o.y, Tf); o.z = __fdiv_rn(o.z, Tf); o.w = __fdiv_rn(o.w, Tf);
      f4_add(sum, o);
    }
    xbin[((size_t)v * rows + r) * e4 + c] = sum;
  }
}

// Frame pooling that also leaves an fp16 copy of the chunk behind (round to nearest even): the short-term attention of
// the caller (Qformer.py:224-304) reads the same tokens as kind::f16 tensor-core operands, so the chunk is streamed
// from HBM once for both (SURVEY 8f N1: "sharing the pass with frame pooling").  Same summation order as pool_unit.
// One (frame, token-split) item: token split sp of frame `src` of the chunk is pooled into row (unit * splits + sp) of
// xpart and converted to the fp16 rows starting at token row `dst16` of k16.
__device__ __forceinline__ void pool_convert_unit_at(const float4* __restrict__ k, float4* __restrict__ xpart,
                                                     uint2* __restrict__ k16, int T, int e4, int splits, float Tf,
                                                     int unit, int sp, size_t src, size_t dst16, uint64_t pol) {
  const int r0 = (int)(((long long)T * sp) / splits);
  const int r1 = (int)(((long long)T * (sp + 1)) / splits);
  const float4* base = k + src * T * e4;
  uint2* base16 = k16 + dst16 * e4;
  // lane pairs (c, c ^ 1) share 16-byte stores when every lane of the warp has a partner inside the row
  // (whole warps only: the exchange is a full-mask shuffle)
  const bool paired = (e4 % 32 == 0) && (reinterpret_cast<uintptr_t>(k16) & 15u) == 0;
  for (int c = threadIdx.x; c < e4; c += blockDim.x) {
    float4 acc[POOL_ACC];
#pragma unroll
    for (int i = 0; i < POOL_ACC; ++i) acc[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    int r = r0;
    for (; r + POOL_UNROLL <= r1; r += POOL_UNROLL) {
      float4 v[POOL_UNROLL];
#pragma unroll
      for (int i = 0; i < POOL_UNROLL; ++i) v[i] = ldg_stream(base + (size_t)(r + i) * e4 + c, pol);
      uint2 pk[POOL_UNROLL];
#pragma unroll
      for (int i = 0; i < POOL_UNROLL; ++i) {
        f4_add(acc[i % POOL_ACC], v[i]);
        const __half2 lo = __floats2half2_rn(v[i].x, v[i].y), hi = __floats2half2_rn(v[i].z, v[i].w);
        pk[i].x = *reinterpret_cast<const uint32_t*>(&lo);
        pk[i].y = *reinterpret_cast<const uint32_t*>(&hi);
      }
      if (paired) {
        // 16-byte stores: neighbouring lanes swap halves of a row pair -- the even lane stores 8 columns of the even
        // row, the odd lane the same 8 columns of the odd row
        const bool odd = (c & 1) != 0;
#pragma unroll
        for (int i = 0; i < POOL_UNROLL; i += 2) {
          const uint2 give = odd ? pk[i] : pk[i + 1];
          uint2 take;
          take.x = __shfl_xor_sync(0xffffffffu, give.x, 1);
          take.y = __shfl_xor_sync(0xffffffffu, give.y, 1);
          const uint2 keep = odd ? pk[i + 1] : pk[i];
          const uint4 out = odd ? make_uint4(take.x, take.y, keep.x, keep.y) : make_uint4(keep.x, keep.y, take.x, take.y);
          *reinterpret_cast<uint4*>(base16 + (size_t)(r + i + (odd ? 1 : 0)) * e4 + (c & ~1)) = out;
        }
      } else {
#pragma unroll
        for (int i = 0; i < POOL_UNROLL; ++i) base16[(size_t)(r + i) * e4 + c] = pk[i];
      }
    }
    for (; r < r1; ++r) {
      const float4 v = ldg_stream(base + (size_t)r * e4 + c, pol);
      f4_add(acc[0], v);
      const __half2 lo = __floats2half2_rn(v.x, v.y), hi = __floats2half2_rn(v.z, v.w);
      uint2 pk;
      pk.x = *reinterpret_cast<const uint32_t*>(&lo);
      pk.y = *reinterpret_cast<const uint32_t*>(&hi);
      base16[(size_t)r * e4 + c] = pk;
    }
#pragma unroll
    for (int i = 1; i < POOL_ACC; ++i) f4_add(acc[0], acc[i]);
    float4 o = acc[0];
    o.x = __fdiv_rn(o.x, Tf); o.y = __fdiv_rn(o.y, Tf); o.z = __fdiv_rn(o.z, Tf); o.w = __fdiv_rn(o.w, Tf);
    xpart[((size_t)unit * splits + sp) * e4 + c] = o;
  }
}

__global__ void __launch_bounds__(256)
pool_mean_convert_kernel(const float4* __restrict__ k, float4* __restrict__ xpart, uint2* __restrict__ k16, int T,
                         int e4, int splits, float Tf) {
  const uint64_t pol = policy_evict_first();
  const unsigned work = blockIdx.x;
  const int unit = work / splits;
  const int sp = work - unit * splits;
  pool_convert_unit_at(k, xpart, k16, T, e4, splits, Tf, unit, sp, (size_t)unit, (size_t)unit * T, pol);
}

// one CTA per (frame, split)
__global__ void __launch_bounds__(256)
pool_mean_kernel(const float4* __restrict__ k, float4* __restrict__ xpart, int T, int e4, int splits, float Tf) {
  pool_unit(k, xpart, T, e4, splits, Tf, blockIdx.x, policy_evict_first());
}

// bounded (persistent) grid walking the work list: leaves SM resources to kernels of other streams while this
// one keeps HBM busy
__global__ void __launch_bounds__(256)
pool_mean_persistent_kernel(const float4* __restrict__ k, float4* __restrict__ xpart, int T, int e4, int splits,
                            float Tf, unsigned total) {
  const uint64_t pol = policy_evict_first();
  for (unsigned work = blockIdx.x; work < total; work += gridDim.x) pool_unit(k, xpart, T, e4, splits, Tf, work, pol);
}

// ---- 16-bit inputs (VideoChat2 runs the Q-former under fp16 autocast, videochat2_it_mistral.py:187): the chunk is
// read as 128-bit vectors of 8 halves / bfloat16s and accumulated in fp32 -- half the HBM bytes of the fp32 path
// and no up-cast pass.  One thread per 8 columns.  Every entry point of the step (plain, prefetched, overlapped, host
// buffers, ragged) pools a 16-bit chunk per frame through pool_unit16_at, so they all give the same bits.
template <bool BF16>
__device__ __forceinline__ void unpack8(const uint4& v, float* f) {
  const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    if (BF16) {
      f[2 * i] = __uint_as_float(w[i] << 16);
      f[2 * i + 1] = __uint_as_float(w[i] & 0xFFFF0000u);
    } else {
      const __half2 h = *reinterpret_cast<const __half2*>(&w[i]);
      const float2 t = __half22float2(h);
      f[2 * i] = t.x;
      f[2 * i + 1] = t.y;
    }
  }
}
__device__ __forceinline__ uint4 ldg_stream_u4(const uint4* p, uint64_t policy) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.u32 {%0,%1,%2,%3}, [%4], %5;"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "l"(p), "l"(policy));
  return r;
}

// 16-bit twin of pool_unit_at
template <bool BF16>
__device__ __forceinline__ void pool_unit16_at(const uint4* __restrict__ k, float4* __restrict__ xpart, int T, int e8,
                                               int splits, float Tf, unsigned unit, int sp, size_t src, uint64_t pol) {
  const int r0 = (int)(((long long)T * sp) / splits);
  const int r1 = (int)(((long long)T * (sp + 1)) / splits);
  const uint4* base = k + src * T * e8;
  for (int c = threadIdx.x; c < e8; c += blockDim.x) {
    float acc[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) acc[i] = 0.f;
    int r = r0;
    for (; r + POOL_UNROLL <= r1; r += POOL_UNROLL) {
      uint4 v[POOL_UNROLL];
#pragma unroll
      for (int i = 0; i < POOL_UNROLL; ++i) v[i] = ldg_stream_u4(base + (size_t)(r + i) * e8 + c, pol);
#pragma unroll
      for (int i = 0; i < POOL_UNROLL; ++i) {
        float f[8];
        unpack8<BF16>(v[i], f);
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[j] += f[j];
      }
    }
    for (; r < r1; ++r) {
      float f[8];
      unpack8<BF16>(ldg_stream_u4(base + (size_t)r * e8 + c, pol), f);
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[j] += f[j];
    }
    float4* dst = xpart + ((size_t)unit * splits + sp) * (2 * e8) + 2 * c;
    dst[0] = make_float4(__fdiv_rn(acc[0], Tf), __fdiv_rn(acc[1], Tf), __fdiv_rn(acc[2], Tf), __fdiv_rn(acc[3], Tf));
    dst[1] = make_float4(__fdiv_rn(acc[4], Tf), __fdiv_rn(acc[5], Tf), __fdiv_rn(acc[6], Tf), __fdiv_rn(acc[7], Tf));
  }
}

// one CTA per (frame, split); PERSIST: bounded grid walking the `total` items (the side-stream pooling of the
// overlapped step), each pooled by the same pool_unit16_at call, so the bits do not depend on the grid
template <bool BF16, bool PERSIST>
__global__ void __launch_bounds__(256)
pool_mean16_kernel(const uint4* __restrict__ k, float4* __restrict__ xpart, int T, int e8, int splits, float Tf,
                   unsigned total) {
  if constexpr (!PERSIST) {
    const unsigned unit = blockIdx.x / splits;
    pool_unit16_at<BF16>(k, xpart, T, e8, splits, Tf, unit, (int)(blockIdx.x - unit * splits), unit,
                         policy_evict_first());
  } else {
    const uint64_t pol = policy_evict_first();
    for (unsigned work = blockIdx.x; work < total; work += gridDim.x) {
      const unsigned unit = work / splits;
      pool_unit16_at<BF16>(k, xpart, T, e8, splits, Tf, unit, (int)(work - unit * splits), unit, pol);
    }
  }
}

template <bool BF16>
static void launch_pool_mean16(const void* k, float* xpart, int T, int e8, int splits, unsigned total, int max_ctas,
                               cudaStream_t st) {
  const int threads = e8 >= 256 ? 256 : ((e8 + 31) / 32) * 32;
  const uint4* k4 = reinterpret_cast<const uint4*>(k);
  float4* x = reinterpret_cast<float4*>(xpart);
  if (max_ctas > 0 && (unsigned)max_ctas < total)
    pool_mean16_kernel<BF16, true><<<(unsigned)max_ctas, threads, 0, st>>>(k4, x, T, e8, splits, (float)T, total);
  else
    pool_mean16_kernel<BF16, false><<<total, threads, 0, st>>>(k4, x, T, e8, splits, (float)T, total);
}

// ---- ragged batch: the grid covers exactly the (frame, token-split) items of the frames in use, packed video after
// video (frame f of the packing is frame f - offs[v] of video v, offs[v] <= f < offs[v+1]); the padding of the chunk
// is never read.  Each item runs the lock-step code above, so a pooled frame carries the same bits.  PERSIST: bounded
// grid walking the item list (the side-stream pooling of step_overlapped).
__device__ __forceinline__ size_t ragged_src(const int32_t* __restrict__ offs, int Bv, int L, unsigned f) {
  int lo = 0, hi = Bv;                                  // offs[lo] <= f < offs[hi]
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if ((unsigned)__ldg(offs + mid) <= f) lo = mid; else hi = mid;
  }
  return (size_t)lo * L + (f - (unsigned)__ldg(offs + lo));
}

template <int DT, bool PERSIST>        // DT: 0 fp32, 1 fp16, 2 bfloat16
__global__ void __launch_bounds__(256)
pool_ragged_kernel(const void* __restrict__ k, float4* __restrict__ xpart, const int32_t* __restrict__ offs, int Bv,
                   int L, int T, int ev, int splits, float Tf, unsigned total) {
  const uint64_t pol = policy_evict_first();
  for (unsigned work = blockIdx.x; work < total; work += gridDim.x) {
    const unsigned f = work / splits;
    const int sp = (int)(work - f * splits);
    const size_t src = ragged_src(offs, Bv, L, f);
    if (DT == 0)
      pool_unit_at(reinterpret_cast<const float4*>(k), xpart, T, ev, splits, Tf, f, sp, src, pol);
    else
      pool_unit16_at<DT == 2>(reinterpret_cast<const uint4*>(k), xpart, T, ev, splits, Tf, f, sp, src, pol);
    if (!PERSIST) break;
  }
}

// Ragged twin of pool_mean_convert_kernel, one CTA per (frame, token-split) item of pool_ragged_kernel: xpart packed
// as there, the fp16 tokens of video v at rows [0, n_v) of its k16 block of ld16 rows (n_v = lengths[v] * T).  The
// last item of a video also zeroes rows [n_v, roundup64(n_v)), so that GEMMs over whole 64-token k-blocks read zeros
// past the video's end; nothing further is written.
__global__ void __launch_bounds__(256)
pool_convert_ragged_kernel(const float4* __restrict__ k, float4* __restrict__ xpart, uint2* __restrict__ k16,
                           const int32_t* __restrict__ offs, int Bv, int L, int T, int e4, int splits, float Tf,
                           long long ld16) {
  const unsigned work = blockIdx.x;
  const unsigned f = work / splits;
  const int sp = (int)(work - f * splits);
  const size_t src = ragged_src(offs, Bv, L, f);
  const int v = (int)(src / L), l = (int)(src - (size_t)v * L);
  pool_convert_unit_at(k, xpart, k16, T, e4, splits, Tf, (int)f, sp, src, (size_t)v * ld16 + (size_t)l * T,
                       policy_evict_first());
  uint2* v16 = k16 + (size_t)v * ld16 * e4;
  if (sp == splits - 1 && f + 1 == (unsigned)__ldg(offs + v + 1)) {
    const int n = (l + 1) * T, n64 = (n + 63) & ~63;
    for (long long i = threadIdx.x; i < (long long)(n64 - n) * e4; i += blockDim.x)
      v16[(size_t)n * e4 + i] = make_uint2(0u, 0u);
  }
}

template <int DT>
static void launch_pool_ragged(const void* k, float* xpart, const int32_t* offs, int Bv, int L, int T, int ev,
                               int splits, float Tf, unsigned total, int max_ctas, cudaStream_t st) {
  const int threads = ev >= 256 ? 256 : ((ev + 31) / 32) * 32;
  float4* x = reinterpret_cast<float4*>(xpart);
  if (max_ctas > 0 && (unsigned)max_ctas < total)
    pool_ragged_kernel<DT, true><<<(unsigned)max_ctas, threads, 0, st>>>(k, x, offs, Bv, L, T, ev, splits, Tf, total);
  else
    pool_ragged_kernel<DT, false><<<total, threads, 0, st>>>(k, x, offs, Bv, L, T, ev, splits, Tf, total);
}

}  // namespace ltm

extern "C" int ltm_pool_mean_ragged(const void* k, int dtype, float* xpart, const int32_t* offs, int Bv, int L, int T,
                                    int e, int splits, int frames, int max_ctas, void* stream) {
  using namespace ltm;
  LTM_REQUIRE(k && xpart && offs, "pool_mean_ragged: null pointer");
  LTM_REQUIRE(Bv > 0 && L > 0 && T > 0 && e > 0 && frames >= 0 && frames <= (long long)Bv * L,
              "pool_mean_ragged: bad shape Bv=%d L=%d T=%d e=%d frames=%d", Bv, L, T, e, frames);
  LTM_REQUIRE(dtype >= 0 && dtype <= 2, "pool_mean_ragged: dtype=%d", dtype);
  LTM_REQUIRE(e % (dtype ? 8 : 4) == 0, "pool_mean_ragged: e=%d must be a multiple of %d", e, dtype ? 8 : 4);
  LTM_REQUIRE(splits >= 1 && splits <= T, "pool_mean_ragged: splits=%d out of range [1,%d]", splits, T);
  LTM_REQUIRE(aligned16(k) && aligned16(xpart), "pool_mean_ragged: pointers must be 16-byte aligned");
  const long long units = (long long)frames * splits;
  LTM_REQUIRE(units < (1ll << 31), "pool_mean_ragged: too many frames");
  if (units == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  const int ev = dtype ? e / 8 : e / 4;
  if (dtype == 0)
    launch_pool_ragged<0>(k, xpart, offs, Bv, L, T, ev, splits, (float)T, (unsigned)units, max_ctas, st);
  else if (dtype == 1)
    launch_pool_ragged<1>(k, xpart, offs, Bv, L, T, ev, splits, (float)T, (unsigned)units, max_ctas, st);
  else
    launch_pool_ragged<2>(k, xpart, offs, Bv, L, T, ev, splits, (float)T, (unsigned)units, max_ctas, st);
  LTM_CHECK_LAUNCH("pool_mean_ragged");
  return 0;
}

extern "C" int ltm_pool_mean_convert_ragged(const float* k, float* xpart, void* k16, const int32_t* offs, int Bv, int L,
                                            int T, int e, int splits, int frames, int ld16, void* stream) {
  using namespace ltm;
  LTM_REQUIRE(k && k16 && offs, "pool_mean_convert_ragged: null pointer");
  LTM_REQUIRE(Bv > 0 && L > 0 && T > 0 && e > 0 && e % 4 == 0 && frames >= 0 && frames <= (long long)Bv * L,
              "pool_mean_convert_ragged: bad shape Bv=%d L=%d T=%d e=%d frames=%d", Bv, L, T, e, frames);
  LTM_REQUIRE(ld16 % 64 == 0 && ld16 >= (long long)L * T,
              "pool_mean_convert_ragged: ld16=%d must be a multiple of 64 and >= L*T=%lld", ld16, (long long)L * T);
  LTM_REQUIRE(splits >= 1 && splits <= T, "pool_mean_convert_ragged: splits=%d out of range [1,%d]", splits, T);
  const long long units = (long long)frames * splits;
  LTM_REQUIRE(units < (1ll << 31), "pool_mean_convert_ragged: too many frames");
  if (units == 0) return 0;                        // every video idle: nothing to read, pool or write (xpart may be NULL)
  LTM_REQUIRE(xpart != nullptr, "pool_mean_convert_ragged: null pointer");
  LTM_REQUIRE(aligned16(k) && aligned16(xpart) && (reinterpret_cast<uintptr_t>(k16) & 7u) == 0,
              "pool_mean_convert_ragged: pointer alignment");
  const int e4 = e / 4;
  const int threads = e4 >= 256 ? 256 : ((e4 + 31) / 32) * 32;
  pool_convert_ragged_kernel<<<(unsigned)units, threads, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<const float4*>(k), reinterpret_cast<float4*>(xpart), reinterpret_cast<uint2*>(k16), offs, Bv, L,
      T, e4, splits, (float)T, (long long)ld16);
  LTM_CHECK_LAUNCH("pool_mean_convert_ragged");
  return 0;
}

extern "C" int ltm_pool_mean_16(const void* k, int is_bf16, float* xpart, int Bv, int L, int T, int e, int splits,
                                void* stream) {
  return ltm_pool_mean_16_grid(k, is_bf16, xpart, Bv, L, T, e, splits, 0, stream);
}

extern "C" int ltm_pool_mean_16_grid(const void* k, int is_bf16, float* xpart, int Bv, int L, int T, int e, int splits,
                                     int max_ctas, void* stream) {
  using namespace ltm;
  LTM_REQUIRE(k && xpart, "pool_mean_16_grid: null pointer");
  LTM_REQUIRE(Bv > 0 && L > 0 && T > 0 && e > 0, "pool_mean_16_grid: bad shape Bv=%d L=%d T=%d e=%d", Bv, L, T, e);
  LTM_REQUIRE(e % 8 == 0, "pool_mean_16_grid: e=%d must be a multiple of 8 (128-bit access of 16-bit elements)", e);
  LTM_REQUIRE(splits >= 1 && splits <= T, "pool_mean_16_grid: splits=%d out of range [1,%d]", splits, T);
  LTM_REQUIRE(max_ctas >= 0, "pool_mean_16_grid: max_ctas=%d must be >= 0", max_ctas);
  LTM_REQUIRE(aligned16(k) && aligned16(xpart), "pool_mean_16_grid: pointers must be 16-byte aligned");
  const long long units = (long long)Bv * L * splits;
  LTM_REQUIRE(units < (1ll << 31), "pool_mean_16_grid: too many frames");
  cudaStream_t st = (cudaStream_t)stream;
  if (is_bf16)
    launch_pool_mean16<true>(k, xpart, T, e / 8, splits, (unsigned)units, max_ctas, st);
  else
    launch_pool_mean16<false>(k, xpart, T, e / 8, splits, (unsigned)units, max_ctas, st);
  LTM_CHECK_LAUNCH("pool_mean_16_grid");
  return 0;
}

extern "C" int ltm_pool_mean(const float* k, float* xpart, int Bv, int L, int T, int e, int splits,
                             void* stream) {
  return ltm_pool_mean_grid(k, xpart, Bv, L, T, e, splits, 0, stream);
}

extern "C" int ltm_pool_mean_grid(const float* k, float* xpart, int Bv, int L, int T, int e, int splits,
                                  int max_ctas, void* stream) {
  using namespace ltm;
  LTM_REQUIRE(k && xpart, "pool_mean: null pointer");
  LTM_REQUIRE(Bv > 0 && L > 0 && T > 0 && e > 0, "pool_mean: bad shape Bv=%d L=%d T=%d e=%d", Bv, L, T, e);
  LTM_REQUIRE(e % 4 == 0, "pool_mean: e=%d must be a multiple of 4 (128-bit access)", e);
  LTM_REQUIRE(splits >= 1 && splits <= T, "pool_mean: splits=%d out of range [1,%d]", splits, T);
  LTM_REQUIRE(aligned16(k) && aligned16(xpart), "pool_mean: pointers must be 16-byte aligned");
  const long long units = (long long)Bv * L * splits;
  LTM_REQUIRE(units < (1ll << 31), "pool_mean: too many frames");
  const int e4 = e / 4;
  const int threads = e4 >= 256 ? 256 : ((e4 + 31) / 32) * 32;
  if (max_ctas > 0 && max_ctas < units) {
    pool_mean_persistent_kernel<<<(unsigned)max_ctas, threads, 0, (cudaStream_t)stream>>>(
        reinterpret_cast<const float4*>(k), reinterpret_cast<float4*>(xpart), T, e4, splits, (float)T, (unsigned)units);
  } else {
    pool_mean_kernel<<<(unsigned)units, threads, 0, (cudaStream_t)stream>>>(
        reinterpret_cast<const float4*>(k), reinterpret_cast<float4*>(xpart), T, e4, splits, (float)T);
  }
  LTM_CHECK_LAUNCH("pool_mean");
  return 0;
}

extern "C" int ltm_pool_bins(const float* k, float* xbin, const int32_t* fbin_ptr, int Bv, int L, int T, int e, int rows,
                             void* stream) {
  using namespace ltm;
  LTM_REQUIRE(k && xbin && fbin_ptr, "pool_bins: null pointer");
  LTM_REQUIRE(Bv > 0 && Bv <= 65535 && L > 0 && T > 0 && e > 0 && e % 4 == 0 && rows > 0,
              "pool_bins: bad shape Bv=%d L=%d T=%d e=%d rows=%d", Bv, L, T, e, rows);
  LTM_REQUIRE(aligned16(k) && aligned16(xbin), "pool_bins: pointers must be 16-byte aligned");
  const int e4 = e / 4;
  const int threads = e4 >= 256 ? 256 : ((e4 + 31) / 32) * 32;
  pool_bins_kernel<<<dim3(rows, Bv), threads, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<const float4*>(k), reinterpret_cast<float4*>(xbin), fbin_ptr, L, T, e4, rows, (float)T);
  LTM_CHECK_LAUNCH("pool_bins");
  return 0;
}

extern "C" int ltm_pool_mean_convert(const float* k, float* xpart, void* k16, int Bv, int L, int T, int e, int splits,
                                     void* stream) {
  using namespace ltm;
  LTM_REQUIRE(k && xpart && k16, "pool_mean_convert: null pointer");
  LTM_REQUIRE(Bv > 0 && L > 0 && T > 0 && e > 0 && e % 4 == 0, "pool_mean_convert: bad shape Bv=%d L=%d T=%d e=%d", Bv, L,
              T, e);
  LTM_REQUIRE(splits >= 1 && splits <= T, "pool_mean_convert: splits=%d out of range [1,%d]", splits, T);
  LTM_REQUIRE(aligned16(k) && aligned16(xpart) && (reinterpret_cast<uintptr_t>(k16) & 7u) == 0,
              "pool_mean_convert: pointer alignment");
  const long long units = (long long)Bv * L * splits;
  LTM_REQUIRE(units < (1ll << 31), "pool_mean_convert: too many frames");
  const int e4 = e / 4;
  const int threads = e4 >= 256 ? 256 : ((e4 + 31) / 32) * 32;
  pool_mean_convert_kernel<<<(unsigned)units, threads, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<const float4*>(k), reinterpret_cast<float4*>(xpart), reinterpret_cast<uint2*>(k16), T, e4, splits,
      (float)T);
  LTM_CHECK_LAUNCH("pool_mean_convert");
  return 0;
}

