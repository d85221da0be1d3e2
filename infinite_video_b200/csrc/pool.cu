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
//
// Every kernel below pools a frame through the pool() of its element type (F32, F16, BF16), so a pooled frame carries
// the same bits whichever kernel, frame map (LockStep, Ragged, PerVideo) or grid produced it.
#include <cuda_fp16.h>
#include <type_traits>

#include "common.cuh"

namespace ltm {

constexpr int POOL_UNROLL = 8;
constexpr int POOL_ACC = 2;

// per-row visitor of F32::mean that does nothing
struct NoVisit {
  template <int N>
  __device__ __forceinline__ void operator()(int, int, const float4 (&)[N]) const {}
};

// ---- element types: one thread owns one 128-bit column group (In) of the chunk.  pool() adds the token rows [r0, r1)
// of one frame for column group c, in the order that defines the type's bits, divides the sums by T and writes them to
// row `row` of xpart.  (Each type computes the store address at its own place on purpose: moving it changes the
// instruction schedule ptxas emits.)  torch.mean == sum / T (true division, so T = 196 rounds like the reference).
// With splits > 1 (small batches only) every partial sum is divided -- and rounded -- on its own and the consumer adds
// the partial means: the pooled frame then differs from sum / T by up to `splits` ulp (1e-7 relative; the coefficient
// tolerance is 1e-5).

// fp32: 8 independent 128-bit loads in flight, folded into two accumulators (the register file is what limits how many
// of these CTAs fit next to the compute-bound kernels of the other stream: 44 registers -> 7 per SM).  visit(r, c, v)
// is handed the rows r, r + 1, ... as they are loaded: 8 at a time, the rows left over one by one.
struct F32 {
  using In = float4;
  template <class Visit>
  static __device__ __forceinline__ float4 mean(const float4* __restrict__ base, int r0, int r1, int e4, int c,
                                                float Tf, uint64_t pol, const Visit& visit) {
    float4 acc[POOL_ACC];
#pragma unroll
    for (int i = 0; i < POOL_ACC; ++i) acc[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    int r = r0;
    for (; r + POOL_UNROLL <= r1; r += POOL_UNROLL) {
      float4 v[POOL_UNROLL];
#pragma unroll
      for (int i = 0; i < POOL_UNROLL; ++i) v[i] = ldg_stream(base + (size_t)(r + i) * e4 + c, pol);
#pragma unroll
      for (int i = 0; i < POOL_UNROLL; ++i) {
        // (packed adds only without a visitor: they tie the rows to register pairs that the fp16 conversion of
        // StoreHalf also needs -- 209 instead of 194 us per 32-video chunk, B200 at 1000 W)
        if constexpr (std::is_same<Visit, NoVisit>::value) f4_add_packed(acc[i % POOL_ACC], v[i]);
        else f4_add(acc[i % POOL_ACC], v[i]);
      }
      visit(r, c, v);
    }
    for (; r < r1; ++r) {
      const float4 v[1] = {ldg_stream(base + (size_t)r * e4 + c, pol)};
      f4_add(acc[0], v[0]);
      visit(r, c, v);
    }
#pragma unroll
    for (int i = 1; i < POOL_ACC; ++i) f4_add(acc[0], acc[i]);
    float4& s = acc[0];
    s.x = __fdiv_rn(s.x, Tf); s.y = __fdiv_rn(s.y, Tf); s.z = __fdiv_rn(s.z, Tf); s.w = __fdiv_rn(s.w, Tf);
    return s;
  }
  template <class Visit>
  static __device__ __forceinline__ void pool(float4* __restrict__ xpart, size_t row, const float4* __restrict__ base,
                                              int r0, int r1, int e4, int c, float Tf, uint64_t pol,
                                              const Visit& visit) {
    const float4 o = mean(base, r0, r1, e4, c, Tf, pol, visit);
    xpart[row * e4 + c] = o;
  }
};

__device__ __forceinline__ uint4 ldg_stream_u4(const uint4* p, uint64_t policy) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.u32 {%0,%1,%2,%3}, [%4], %5;"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "l"(p), "l"(policy));
  return r;
}

// 16-bit inputs (VideoChat2 runs the Q-former under fp16 autocast, videochat2_it_mistral.py:187): the chunk is read as
// 128-bit vectors of 8 halves / bfloat16s and accumulated in fp32, rows in order -- half the HBM bytes of the fp32
// path and no up-cast pass.  One thread per 8 columns.
template <bool IS_BF16>
struct Half {
  using In = uint4;
  static __device__ __forceinline__ void unpack8(const uint4& v, float* f) {
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      if (IS_BF16) {
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
  static __device__ __forceinline__ void pool(float4* __restrict__ xpart, size_t row, const uint4* __restrict__ base,
                                              int r0, int r1, int e8, int c, float Tf, uint64_t pol, NoVisit) {
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
        unpack8(v[i], f);
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[j] += f[j];
      }
    }
    for (; r < r1; ++r) {
      float f[8];
      unpack8(ldg_stream_u4(base + (size_t)r * e8 + c, pol), f);
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[j] += f[j];
    }
    float4* dst = xpart + row * (2 * e8) + 2 * c;
    dst[0] = make_float4(__fdiv_rn(acc[0], Tf), __fdiv_rn(acc[1], Tf), __fdiv_rn(acc[2], Tf), __fdiv_rn(acc[3], Tf));
    dst[1] = make_float4(__fdiv_rn(acc[4], Tf), __fdiv_rn(acc[5], Tf), __fdiv_rn(acc[6], Tf), __fdiv_rn(acc[7], Tf));
  }
};
using F16 = Half<false>;
using BF16 = Half<true>;

// ---- frame maps: the work items are the (frame, token-split) pairs of the pooled frames, frame f of them read from
// frame src(f) of the chunk, which starts at frame(k, src(f), T, ev).  A kernel builds its map from its last three
// arguments: offs[Bv+1], Bv, L.  (Scalar arguments rather than a struct: a struct argument is loaded whole and held in
// registers across the work loop.)
struct LockStep {      // every video uses all L frames: frame v*L + l in and out
  static constexpr bool ragged = false;
  __device__ __forceinline__ LockStep(const int32_t*, int, int) {}
  __device__ __forceinline__ size_t src(unsigned f) const { return f; }
  template <class In>
  static __device__ __forceinline__ const In* frame(const In* k, size_t src, int T, int ev) { return k + src * T * ev; }
};
struct Ragged {        // frames packed video after video: frame f is frame f - offs[v] of video v, offs[v] <= f <
  static constexpr bool ragged = true;     // offs[v+1]; the padding of the chunk is never read
  const int32_t* offs;
  int Bv, L;
  __device__ __forceinline__ int video(unsigned f) const {
    int lo = 0, hi = Bv;                                  // offs[lo] <= f < offs[hi]
    while (hi - lo > 1) {
      const int mid = (lo + hi) >> 1;
      if ((unsigned)__ldg(offs + mid) <= f) lo = mid; else hi = mid;
    }
    return lo;
  }
  __device__ __forceinline__ size_t src(unsigned f) const {
    const int v = video(f);
    return (size_t)v * L + (f - (unsigned)__ldg(offs + v));
  }
  template <class In>
  static __device__ __forceinline__ const In* frame(const In* k, size_t src, int T, int ev) { return k + src * T * ev; }
};
// The work items of Ragged, each video's frames read from wherever its chunk lives: k is then a table of Bv 64-bit
// base addresses, and frame l of video v starts at ptrs[v] + l*T*e.  src(f) packs (v, l) as v << 32 | l.  (The
// offset in a video is a 32-bit product, L*T*ev < 2^32 is checked on the host: with a 64-bit one the bounded-grid
// 16-bit kernels spill.)
struct PerVideo : Ragged {
  __device__ __forceinline__ PerVideo(const int32_t* o, int b, int l) : Ragged{o, b, l} {}
  __device__ __forceinline__ size_t src(unsigned f) const {
    const int v = video(f);
    return (size_t)v << 32 | (f - (unsigned)__ldg(offs + v));
  }
  template <class In>
  static __device__ __forceinline__ const In* frame(const In* k, size_t src, int T, int ev) {
    const auto* ptrs = reinterpret_cast<const unsigned long long*>(k);
    return reinterpret_cast<const In*>(__ldg(ptrs + (src >> 32))) + (size_t)((unsigned)src * (unsigned)(T * ev));
  }
};

struct WorkItem {
  unsigned f;          // pooled frame
  int sp;              // token split
  size_t src;          // frame of the chunk
};
template <class Map>
__device__ __forceinline__ WorkItem work_item(const Map& map, unsigned work, int splits) {
  const unsigned f = work / splits;
  return {f, (int)(work - f * splits), map.src(f)};
}

// Token split it.sp of chunk frame it.src, written to row (it.f * splits + it.sp) of xpart.
template <class E, class Map, class Visit = NoVisit>
__device__ __forceinline__ void pool_item(const typename E::In* __restrict__ k, float4* __restrict__ xpart, int T,
                                          int ev, int splits, float Tf, const WorkItem& it, uint64_t pol,
                                          const Visit& visit = {}) {
  const int r0 = (int)(((long long)T * it.sp) / splits);
  const int r1 = (int)(((long long)T * (it.sp + 1)) / splits);
  const typename E::In* base = Map::frame(k, it.src, T, ev);
  for (int c = threadIdx.x; c < ev; c += blockDim.x)
    E::pool(xpart, (size_t)it.f * splits + it.sp, base, r0, r1, ev, c, Tf, pol, visit);
}

// One CTA per work item; PERSIST: a bounded grid walking the `total` items, which leaves SM resources to the kernels
// of other streams while this one keeps HBM busy (the side-stream pooling of step_overlapped).
template <class E, class Map, bool PERSIST>
__global__ void __launch_bounds__(256)
pool_mean_kernel(const typename E::In* __restrict__ k, float4* __restrict__ xpart, int T, int ev, int splits,
                 float Tf, unsigned total, const int32_t* offs, int Bv, int L) {
  const Map map{offs, Bv, L};
  if constexpr (!PERSIST) {
    pool_item<E, Map>(k, xpart, T, ev, splits, Tf, work_item(map, blockIdx.x, splits), policy_evict_first());
  } else {
    const uint64_t pol = policy_evict_first();
    for (unsigned work = blockIdx.x; work < total; work += gridDim.x)
      pool_item<E, Map>(k, xpart, T, ev, splits, Tf, work_item(map, work, splits), pol);
  }
}

// Frame pooling folded with the first half of the regression (VERDICT r1, "bin sums instead of xpart"): the frames of
// an update chunk that fall into the same basis bin are consecutive (tables.py: fbin_ptr), and the consolidation only
// ever needs their sum, so one CTA per (video, bin) pools its frames one after the other -- each exactly like
// pool_mean_kernel with splits == 1 -- and writes the running sum of the frame means: xbin[v, r, :] = sum_f mean_t
// k[v,f,t,:].  At the NExT-QA shape that is 64 rows per video instead of 256 (0.2 instead of 0.8 MB written and read
// back).  (Measured alternatives: FP = 2..4 frames of a bin side by side in one CTA of FP x 192 threads, frame means
// staged in shared memory.  Alone on the GPU that is the fastest pooling kernel of all -- 0.4645 ms for 3.2 GB at
// FP = 4 -- but next to the other stream's kernels its large CTAs lose: 188.6 k chunks/s at FP = 4, 192.9 k at
// FP = 2, against 194.4 k for this one-frame-at-a-time form, whose CTAs hold 7.7 k registers each and leave room
// sooner.)
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
      f4_add(sum, F32::mean(kv + (size_t)f * T * e4, 0, T, e4, c, Tf, pol, NoVisit{}));
    }
    xbin[((size_t)v * rows + r) * e4 + c] = sum;
  }
}

// Per-row visitor of F32::mean that stores every row it is handed as fp16 (round to nearest even) at row r of base16.
struct StoreHalf {
  uint2* base16;
  int e4;
  // lane pairs (c, c ^ 1) share 16-byte stores when every lane of the warp has a partner inside the row
  // (whole warps only: the exchange is a full-mask shuffle)
  bool paired;
  template <int N>
  __device__ __forceinline__ void operator()(int r, int c, const float4 (&v)[N]) const {
    uint2 pk[N];
#pragma unroll
    for (int i = 0; i < N; ++i) {
      const __half2 lo = __floats2half2_rn(v[i].x, v[i].y), hi = __floats2half2_rn(v[i].z, v[i].w);
      pk[i].x = *reinterpret_cast<const uint32_t*>(&lo);
      pk[i].y = *reinterpret_cast<const uint32_t*>(&hi);
    }
    // (addresses stepped from one row pointer: 64-bit products per row leave both convert kernels spilling)
    uint2* row = base16 + (size_t)r * e4;
    if constexpr (N % 2 == 0) {
      if (paired) {
        // 16-byte stores: neighbouring lanes swap halves of a row pair -- the even lane stores 8 columns of the even
        // row, the odd lane the same 8 columns of the odd row
        const bool odd = (c & 1) != 0;
        uint2* p = row + (odd ? e4 : 0) + (c & ~1);
#pragma unroll
        for (int i = 0; i < N; i += 2) {
          const uint2 give = odd ? pk[i] : pk[i + 1];
          uint2 take;
          take.x = __shfl_xor_sync(0xffffffffu, give.x, 1);
          take.y = __shfl_xor_sync(0xffffffffu, give.y, 1);
          const uint2 keep = odd ? pk[i + 1] : pk[i];
          const uint4 out = odd ? make_uint4(take.x, take.y, keep.x, keep.y) : make_uint4(keep.x, keep.y, take.x, take.y);
          *reinterpret_cast<uint4*>(p) = out;
          p += 2 * e4;
        }
        return;
      }
    }
    row += c;
#pragma unroll
    for (int i = 0; i < N; ++i, row += e4) *row = pk[i];
  }
};

// Frame pooling that also leaves an fp16 copy of the chunk behind: the short-term attention of the caller
// (Qformer.py:224-304) reads the same tokens as kind::f16 tensor-core operands, so the chunk is streamed from HBM once
// for both (SURVEY 8f N1: "sharing the pass with frame pooling").  One CTA per work item of pool_mean_kernel.  k16 is
// the chunk's own shape for LockStep; for Ragged, the tokens of video v sit at rows [0, n_v) of its k16 block of ld16
// rows (n_v = lengths[v] * T), and the last item of a video also zeroes rows [n_v, roundup64(n_v)), so that GEMMs over
// whole 64-token k-blocks read zeros past the video's end; nothing further is written.
template <class Map>
__global__ void __launch_bounds__(256)
pool_mean_convert_kernel(const float4* __restrict__ k, float4* __restrict__ xpart, uint2* __restrict__ k16, int T,
                         int e4, int splits, float Tf, long long ld16, const int32_t* offs, int Bv, int L) {
  const Map map{offs, Bv, L};
  const WorkItem it = work_item(map, blockIdx.x, splits);
  const bool paired = (e4 % 32 == 0) && (reinterpret_cast<uintptr_t>(k16) & 15u) == 0;
  size_t row16 = it.src * T;
  if constexpr (Map::ragged) {       // (the tail first: v and l are then not held through the pooling loop)
    const int v = (int)(it.src / L), l = (int)(it.src - (size_t)v * L);
    row16 = (size_t)v * ld16 + (size_t)l * T;
    if (it.sp == splits - 1 && it.f + 1 == (unsigned)__ldg(offs + v + 1)) {
      uint2* v16 = k16 + (size_t)v * ld16 * e4;
      const int n = (l + 1) * T, n64 = (n + 63) & ~63;
      for (long long i = threadIdx.x; i < (long long)(n64 - n) * e4; i += blockDim.x)
        v16[(size_t)n * e4 + i] = make_uint2(0u, 0u);
    }
  }
  pool_item<F32, Map>(k, xpart, T, e4, splits, Tf, it, policy_evict_first(), StoreHalf{k16 + row16 * e4, e4, paired});
}

template <class Map, class E>
static void launch_mean(const void* k, float* xpart, const int32_t* offs, int Bv, int L, int T, int ev, int splits,
                        unsigned units, int max_ctas, int threads, cudaStream_t st) {
  const auto* kk = reinterpret_cast<const typename E::In*>(k);
  float4* x = reinterpret_cast<float4*>(xpart);
  if (max_ctas > 0 && (unsigned)max_ctas < units)
    pool_mean_kernel<E, Map, true><<<(unsigned)max_ctas, threads, 0, st>>>(kk, x, T, ev, splits, (float)T, units, offs,
                                                                          Bv, L);
  else
    pool_mean_kernel<E, Map, false><<<units, threads, 0, st>>>(kk, x, T, ev, splits, (float)T, units, offs, Bv, L);
}

template <class Map>
static void launch_mean(int dtype, const void* k, float* xpart, const int32_t* offs, int Bv, int L, int T, int ev,
                        int splits, unsigned units, int max_ctas, int threads, cudaStream_t st) {
  if (dtype == 0)
    launch_mean<Map, F32>(k, xpart, offs, Bv, L, T, ev, splits, units, max_ctas, threads, st);
  else if (dtype == 1)
    launch_mean<Map, F16>(k, xpart, offs, Bv, L, T, ev, splits, units, max_ctas, threads, st);
  else
    launch_mean<Map, BF16>(k, xpart, offs, Bv, L, T, ev, splits, units, max_ctas, threads, st);
}

int pool_frames(const char* who, const void* k, int dtype, float* xpart, int Bv, int L, int T, int e, int splits,
                int max_ctas, void* stream, const int32_t* offs, int frames, void* k16, int ld16,
                const int32_t* fbin_ptr, int rows, const void* const* ptrs) {
  const long long nf = offs ? frames : (long long)Bv * L, units = nf * splits;
  LTM_REQUIRE((k || ptrs) && (xpart || units == 0), "%s: null pointer", who);
  LTM_REQUIRE(!ptrs || (offs && !k && !k16 && !fbin_ptr),
              "%s: a chunk pointer table needs frame offsets and takes no chunk, fp16 copy or per-bin pooling", who);
  LTM_REQUIRE(Bv > 0 && L > 0 && T > 0 && e > 0 && nf >= 0 && nf <= (long long)Bv * L &&
              (!fbin_ptr || (rows > 0 && Bv <= 65535)),
              "%s: bad shape Bv=%d L=%d T=%d e=%d frames=%lld rows=%d", who, Bv, L, T, e, nf, rows);
  LTM_REQUIRE(dtype >= 0 && dtype <= 2, "%s: dtype=%d", who, dtype);
  const int w = dtype ? 8 : 4;                               // elements per 128-bit column group
  LTM_REQUIRE(e % w == 0, "%s: e=%d must be a multiple of %d (128-bit access)", who, e, w);
  LTM_REQUIRE(!(k16 && offs) || (ld16 % 64 == 0 && ld16 >= (long long)L * T),
              "%s: ld16=%d must be a multiple of 64 and >= L*T=%lld", who, ld16, (long long)L * T);
  LTM_REQUIRE(splits >= 1 && splits <= T, "%s: splits=%d out of range [1,%d]", who, splits, T);
  LTM_REQUIRE(max_ctas >= 0, "%s: max_ctas=%d must be >= 0", who, max_ctas);
  LTM_REQUIRE(aligned16(k) && aligned16(xpart) && (reinterpret_cast<uintptr_t>(k16) & 7u) == 0 &&
              (reinterpret_cast<uintptr_t>(ptrs) & 7u) == 0,
              "%s: pointers must be 16-byte aligned%s", who, k16 ? " (k16: 8-byte)" : ptrs ? " (ptrs: 8-byte)" : "");
  LTM_REQUIRE(units < (1ll << 31), "%s: too many frames", who);
  LTM_REQUIRE(!ptrs || (long long)L * T * (e / w) < (1ll << 32), "%s: a video of L*T*e=%lld elements is too large for "
              "the pointer table", who, (long long)L * T * e);
  if (units == 0) return 0;                  // every video of a ragged chunk idle: nothing to read, pool or write
  const int ev = e / w;
  const int threads = ev >= 256 ? 256 : ((ev + 31) / 32) * 32;
  cudaStream_t st = (cudaStream_t)stream;
  const float4* k4 = reinterpret_cast<const float4*>(k);
  float4* x4 = reinterpret_cast<float4*>(xpart);
  uint2* h = reinterpret_cast<uint2*>(k16);
  if (fbin_ptr)
    pool_bins_kernel<<<dim3(rows, Bv), threads, 0, st>>>(k4, x4, fbin_ptr, L, T, ev, rows, (float)T);
  else if (k16 && offs)
    pool_mean_convert_kernel<Ragged><<<(unsigned)units, threads, 0, st>>>(k4, x4, h, T, ev, splits, (float)T, ld16,
                                                                           offs, Bv, L);
  else if (k16)
    pool_mean_convert_kernel<LockStep><<<(unsigned)units, threads, 0, st>>>(k4, x4, h, T, ev, splits, (float)T, 0,
                                                                             offs, Bv, L);
  else if (ptrs)
    launch_mean<PerVideo>(dtype, ptrs, xpart, offs, Bv, L, T, ev, splits, (unsigned)units, max_ctas, threads, st);
  else if (offs)
    launch_mean<Ragged>(dtype, k, xpart, offs, Bv, L, T, ev, splits, (unsigned)units, max_ctas, threads, st);
  else
    launch_mean<LockStep>(dtype, k, xpart, offs, Bv, L, T, ev, splits, (unsigned)units, max_ctas, threads, st);
  LTM_CHECK_LAUNCH(who);
  return 0;
}

}  // namespace ltm

extern "C" int ltm_pool_mean(const float* k, float* xpart, int Bv, int L, int T, int e, int splits, void* stream) {
  return ltm_pool_mean_grid(k, xpart, Bv, L, T, e, splits, 0, stream);
}

extern "C" int ltm_pool_mean_grid(const float* k, float* xpart, int Bv, int L, int T, int e, int splits,
                                  int max_ctas, void* stream) {
  return ltm::pool_frames("pool_mean", k, 0, xpart, Bv, L, T, e, splits, max_ctas, stream);
}

extern "C" int ltm_pool_mean_16(const void* k, int is_bf16, float* xpart, int Bv, int L, int T, int e, int splits,
                                void* stream) {
  return ltm_pool_mean_16_grid(k, is_bf16, xpart, Bv, L, T, e, splits, 0, stream);
}

extern "C" int ltm_pool_mean_16_grid(const void* k, int is_bf16, float* xpart, int Bv, int L, int T, int e, int splits,
                                     int max_ctas, void* stream) {
  return ltm::pool_frames("pool_mean_16_grid", k, is_bf16 ? 2 : 1, xpart, Bv, L, T, e, splits, max_ctas, stream);
}

extern "C" int ltm_pool_mean_ragged(const void* k, int dtype, float* xpart, const int32_t* offs, int Bv, int L, int T,
                                    int e, int splits, int frames, int max_ctas, void* stream) {
  LTM_REQUIRE(offs, "pool_mean_ragged: null pointer");
  return ltm::pool_frames("pool_mean_ragged", k, dtype, xpart, Bv, L, T, e, splits, max_ctas, stream, offs, frames);
}

extern "C" int ltm_pool_mean_ptrs(const void* const* ptrs, int dtype, float* xpart, const int32_t* offs, int Bv, int L,
                                  int T, int e, int splits, int frames, int max_ctas, void* stream) {
  LTM_REQUIRE(ptrs && offs, "pool_mean_ptrs: null pointer");
  return ltm::pool_frames("pool_mean_ptrs", nullptr, dtype, xpart, Bv, L, T, e, splits, max_ctas, stream, offs, frames,
                          nullptr, 0, nullptr, 0, ptrs);
}

extern "C" int ltm_pool_mean_convert(const float* k, float* xpart, void* k16, int Bv, int L, int T, int e, int splits,
                                     void* stream) {
  LTM_REQUIRE(k16, "pool_mean_convert: null pointer");
  return ltm::pool_frames("pool_mean_convert", k, 0, xpart, Bv, L, T, e, splits, 0, stream, nullptr, 0, k16);
}

extern "C" int ltm_pool_mean_convert_ragged(const float* k, float* xpart, void* k16, const int32_t* offs, int Bv, int L,
                                            int T, int e, int splits, int frames, int ld16, void* stream) {
  LTM_REQUIRE(k16 && offs, "pool_mean_convert_ragged: null pointer");
  return ltm::pool_frames("pool_mean_convert_ragged", k, 0, xpart, Bv, L, T, e, splits, 0, stream, offs, frames, k16,
                          ld16);
}

extern "C" int ltm_pool_bins(const float* k, float* xbin, const int32_t* fbin_ptr, int Bv, int L, int T, int e, int rows,
                             void* stream) {
  LTM_REQUIRE(fbin_ptr, "pool_bins: null pointer");
  return ltm::pool_frames("pool_bins", k, 0, xbin, Bv, L, T, e, 1, 0, stream, nullptr, 0, nullptr, 0, fbin_ptr, rows);
}
