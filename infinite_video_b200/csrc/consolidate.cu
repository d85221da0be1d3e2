// R3/R5/R8 -- memory contraction + ridge regression for rectangular bases
// (long_term_attention_gibbs.py:184-222, compute_G :68-84).
//
// With indicator bases F F^T is diagonal, so G = F^T (F F^T + 0.5 I)^-1 has one non-zero per row,
// 1/(cnt_j + 0.5), and  B = G^T [xm ; x]  is a segmented mean over the (contiguous) positions that
// fall into bin j: contracted re-samples of the old memory -- rows of B_past gathered through the
// sticky sample indices, i.e. the one-hot product B_past^T Psi^T of :208-210 -- followed by the
// new pooled frames.  One CTA produces one coefficient row (four in a row for large batches); one thread one 128-bit
// column group.
#include <cuda_fp16.h>

#include "common.cuh"

namespace ltm {

struct KvState {
  const float4* KV_past;      // [Bv, N, ldkv4] previous call's K|V (NULL: coefficients only)
  float4* KV_new;
  const float4* bkv;          // [ldkv4]
  int ldkv4, jf, round_tf32;
  int half;                   // K|V are stored as IEEE fp16 ([Bv, N, ldkv] halves): same pointers, read as uint4 = 8 halves
};

__device__ __forceinline__ float tf32_round(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return __uint_as_float(r);
}

// Ragged batch (RAGGED kernels only): video v has lengths[v] frames, packed from frame offs[v] in xpart; its tables are
// entry lengths[v] of the table bank (seg_ptr0/1 [L+1, N+1] with absolute member offsets, g0/1 [L+1, N]).  An idle
// video (lengths[v] == 0) keeps its coefficients: B_past is copied to B_new (zeros for a slot that holds no memory,
// B_past == NULL) together with the fp16 copy, so that every later kernel of the call sees defined operands for it.
struct Ragged {
  const int32_t* lengths;
  const int32_t* offs;
};

template <int ROWS, bool RAGGED>
__global__ void __launch_bounds__(256)
consolidate_rect_kernel(const float4* __restrict__ B_past, const float4* __restrict__ xpart,
                        const int32_t* __restrict__ idx, const long long idx_stride,
                        const uint8_t* __restrict__ new_doc,
                        const int32_t* __restrict__ seg_ptr0, const int32_t* __restrict__ seg_mem0,
                        const float* __restrict__ g0,
                        const int32_t* __restrict__ seg_ptr1, const int32_t* __restrict__ seg_mem1,
                        const float* __restrict__ g1,
                        float4* __restrict__ B_new, uint2* __restrict__ B_half, const KvState kv, int N, int e4, int L,
                        int splits, int S, const Ragged rg) {
  const int v = blockIdx.y;
  long long xrow = (long long)v * L;          // first pooled frame of this video in xpart
  if (RAGGED) {
    const int Lv = rg.lengths[v];
    if (Lv == 0) {
#pragma unroll 1
      for (int jr = 0; jr < ROWS; ++jr) {
        const int j = blockIdx.x * ROWS + jr;
        if (j >= N) break;
        for (int c = threadIdx.x; c < e4; c += blockDim.x) {
          const size_t o = ((size_t)v * N + j) * e4 + c;
          const float4 b = B_past != nullptr ? B_past[o] : make_float4(0.f, 0.f, 0.f, 0.f);
          B_new[o] = b;
          if (B_half != nullptr) {
            const __half2 lo = __floats2half2_rn(b.x, b.y), hi = __floats2half2_rn(b.z, b.w);
            B_half[o] = make_uint2(*reinterpret_cast<const uint32_t*>(&lo), *reinterpret_cast<const uint32_t*>(&hi));
          }
        }
      }
      return;
    }
    xrow = rg.offs[v];
    seg_ptr0 += (size_t)Lv * (N + 1); g0 += (size_t)Lv * N;
    seg_ptr1 += (size_t)Lv * (N + 1); g1 += (size_t)Lv * N;
  }
  // ROWS coefficient rows per CTA (1: the loop folds away and the kernel is the one-row kernel, 32 registers)
#pragma unroll 1
  for (int jr = 0; jr < ROWS; ++jr) {
  const int j = blockIdx.x * ROWS + jr;
  if (ROWS > 1 && j >= N) break;
  const bool first = (B_past == nullptr) || (new_doc != nullptr && new_doc[v] != 0);
  const int32_t* seg_ptr = first ? seg_ptr0 : seg_ptr1;
  const int32_t* seg_mem = first ? seg_mem0 : seg_mem1;
  const float g = first ? g0[j] : g1[j];
  const int m0 = seg_ptr[j], m1 = seg_ptr[j + 1];
  const int frame_base = first ? 0 : S;       // member ids >= frame_base are frames
  const float4* xv = xpart + (size_t)xrow * splits * e4;
  const float4* bv = first ? nullptr : B_past + (size_t)v * N * e4;
  const int32_t* iv = first ? nullptr : idx + (size_t)v * idx_stride;
  for (int c = threadIdx.x; c < e4; c += blockDim.x) {
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int m = m0; m < m1; ++m) {
      const int p = seg_mem[m];
      if (p >= frame_base) {
        const float4* src = xv + (size_t)(p - frame_base) * splits * e4 + c;
        for (int s = 0; s < splits; ++s) f4_add(acc, src[(size_t)s * e4]);
      } else {
        const int row = iv[p];
        if (row >= 0) f4_add(acc, bv[(size_t)row * e4 + c]);
      }
    }
    acc.x *= g; acc.y *= g; acc.z *= g; acc.w *= g;
    B_new[((size_t)v * N + j) * e4 + c] = acc;
    // fp16 copy: operand of the K/V projection (kind::f16 UMMAs) -- only the rows the projection will read
    if (B_half != nullptr && (kv.KV_past == nullptr || first || j >= kv.jf)) {
      const __half2 lo = __floats2half2_rn(acc.x, acc.y), hi = __floats2half2_rn(acc.z, acc.w);
      uint2 pk;
      pk.x = *reinterpret_cast<const uint32_t*>(&lo);
      pk.y = *reinterpret_cast<const uint32_t*>(&hi);
      B_half[((size_t)v * N + j) * e4 + c] = pk;
    }
  }
  // projected memory: a bin below jf holds re-sampled memory only, and K|V = B W^T + b is affine in B, so its
  // keys / values are the same segmented mean taken over the previous call's K|V rows (the bias enters once:
  // g sum_p (KV_past[p] - b) + b).  Rows >= jf are left to the projection GEMM.
  if (kv.KV_past != nullptr && !first && j < kv.jf && kv.half) {
    // fp16 K|V: rows of ldkv4 * 4 halves = ldkv8 uint4; fp32 accumulation, one rounding at the store
    const int ld8 = kv.ldkv4 / 2;
    const uint4* kvp = reinterpret_cast<const uint4*>(kv.KV_past) + (size_t)v * N * ld8;
    uint4* out = reinterpret_cast<uint4*>(kv.KV_new) + ((size_t)v * N + j) * ld8;
    int cnt = 0;
    for (int m = m0; m < m1; ++m) cnt += (iv[seg_mem[m]] >= 0) ? 1 : 0;
    const float bw = 1.f - g * (float)cnt;
    for (int c = threadIdx.x; c < ld8; c += blockDim.x) {
      float acc[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) acc[i] = 0.f;
      for (int m = m0; m < m1; ++m) {
        const int row = iv[seg_mem[m]];
        if (row >= 0) {
          const uint4 u = kvp[(size_t)row * ld8 + c];
          const uint32_t w4[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&w4[i]));
            acc[2 * i] += f.x;
            acc[2 * i + 1] += f.y;
          }
        }
      }
      const float4 b0 = kv.bkv[2 * c], b1 = kv.bkv[2 * c + 1];
      const float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
      uint32_t pk[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const __half2 h = __floats2half2_rn(fmaf(acc[2 * i], g, bw * bb[2 * i]), fmaf(acc[2 * i + 1], g, bw * bb[2 * i + 1]));
        pk[i] = *reinterpret_cast<const uint32_t*>(&h);
      }
      out[c] = make_uint4(pk[0], pk[1], pk[2], pk[3]);
    }
  } else if (kv.KV_past != nullptr && !first && j < kv.jf) {
    const float4* kvp = kv.KV_past + (size_t)v * N * kv.ldkv4;
    int cnt = 0;
    for (int m = m0; m < m1; ++m) cnt += (iv[seg_mem[m]] >= 0) ? 1 : 0;
    const float bw = 1.f - g * (float)cnt;
    for (int c = threadIdx.x; c < kv.ldkv4; c += blockDim.x) {
      float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
      for (int m = m0; m < m1; ++m) {
        const int row = iv[seg_mem[m]];
        if (row >= 0) f4_add(acc, kvp[(size_t)row * kv.ldkv4 + c]);
      }
      const float4 b = kv.bkv[c];
      acc.x = fmaf(acc.x, g, bw * b.x); acc.y = fmaf(acc.y, g, bw * b.y);
      acc.z = fmaf(acc.z, g, bw * b.z); acc.w = fmaf(acc.w, g, bw * b.w);
      if (kv.round_tf32) acc = make_float4(tf32_round(acc.x), tf32_round(acc.y), tf32_round(acc.z), tf32_round(acc.w));
      kv.KV_new[((size_t)v * N + j) * kv.ldkv4 + c] = acc;
    }
  }
  }   // rows of this CTA
}

// Variant G, sticky update: the S re-sampled rows xm[s] = R[b_s] (R = Psi_tab B_past, 128 candidate rows) enter the
// regression as G_inf^T[:, :S] xm = sum_b (sum_{s: b_s = b} G_inf^T[:, s]) R[b]: with the draws sorted by bin the inner
// sums are runs of consecutive columns of the (constant) operator.  out[v, n, b] = sum of GT[n, s] over the run of bin b,
// out[v, n, nbins + l] = GT[n, S + l] (the frame columns, copied): a per-video operator with 128 + L instead of S + L
// columns whose product with [R ; k] is the same B -- without materialising xm[Bv, S, e] and with half the
// contraction length.  long_term_attention.py:239-250.
// One warp per operator row: the S sample columns are read 32 at a time (coalesced) next to their (sorted) bins, a
// segmented warp scan adds the members of a bin that sit in the same 32, and the last lane of each segment adds the
// partial to the row's per-bin accumulator in shared memory -- a long run (a peaky histogram puts a hundred draws into
// one bin) costs what a short one does.
constexpr int FOLD_UNROLL = 8;
__global__ void __launch_bounds__(256)
fold_sample_columns_kernel(const float* __restrict__ GT, long long ldg, const int32_t* __restrict__ b_sorted,
                           float* __restrict__ out, int N, int S, int L, int nbins, int rows_per_cta) {
  extern __shared__ float facc[];                          // [8 warps][nbins]
  const int v = blockIdx.y, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int32_t* bs = b_sorted + (size_t)v * S;
  float* acc = facc + warp * nbins;
  const int W = nbins + L;
  for (int r = warp; r < rows_per_cta; r += 8) {
    const int n = blockIdx.x * rows_per_cta + r;
    if (n >= N) break;                                     // warp-uniform
    const float* g = GT + (size_t)n * ldg;
    for (int b = lane; b < nbins; b += 32) acc[b] = 0.f;
    __syncwarp();
    for (int s0 = 0; s0 < S; s0 += 32 * FOLD_UNROLL) {
      // the loads of FOLD_UNROLL chunks go out together (the loop is bound by their latency, not by the arithmetic)
      int key[FOLD_UNROLL];
      float val[FOLD_UNROLL];
#pragma unroll
      for (int u = 0; u < FOLD_UNROLL; ++u) {
        const int s = s0 + 32 * u + lane;
        key[u] = s < S ? __ldg(bs + s) : -1 - lane;        // (padding lanes: unique keys, nothing to add)
        val[u] = s < S ? __ldg(g + s) : 0.f;
      }
#pragma unroll
      for (int u = 0; u < FOLD_UNROLL; ++u) {
        const int s = s0 + 32 * u + lane;
        // segmented inclusive scan over equal (sorted, hence adjacent) keys
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const float up = __shfl_up_sync(0xffffffffu, val[u], o);
          const int ku = __shfl_up_sync(0xffffffffu, key[u], o);
          if (lane >= o && ku == key[u]) val[u] += up;
        }
        const int kn = __shfl_down_sync(0xffffffffu, key[u], 1);
        if (s < S && (lane == 31 || kn != key[u]) && key[u] >= 0 && key[u] < nbins) acc[key[u]] += val[u];
        __syncwarp();                                      // segment tails of one chunk hit distinct bins
      }
    }
    float* o = out + ((size_t)v * N + n) * W;
    for (int b = lane; b < nbins; b += 32) o[b] = acc[b];
    for (int l = lane; l < L; l += 32) o[nbins + l] = g[S + l];
    __syncwarp();
  }
}

// Idle videos of a ragged batch: dst[v] = src[v] (zero when src == NULL) for every v with lengths[v] == 0, as n words
// of type W per video.  Keeps what an idle video owns -- coefficient rows, K|V rows, sticky histogram partials -- bit
// for bit across a call whose kernels run over every video, and zeroes its ctx rows.
template <class W>
__global__ void __launch_bounds__(256)
carry_idle_kernel(const int32_t* __restrict__ lengths, const W* __restrict__ src, W* __restrict__ dst, long long n) {
  const int v = blockIdx.y;
  if (lengths[v] != 0) return;
  const W* s = src ? src + (size_t)v * n : nullptr;
  W* d = dst + (size_t)v * n;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    d[i] = s ? s[i] : W{};
}

int carry_idle(const int32_t* lengths, const void* src, void* dst, size_t bytes_per_video, int Bv, void* stream) {
  LTM_REQUIRE(lengths && dst && bytes_per_video % 4 == 0 && Bv <= 65535, "carry_idle: bad arguments");
  // 16-byte words where every video's slice is 16-byte aligned, else 4-byte words
  const bool wide = bytes_per_video % 16 == 0 && aligned16(src) && aligned16(dst);
  const long long n = (long long)(bytes_per_video / (wide ? 16 : 4));
  const int blocks = (int)((n + 255) / 256 < 64 ? (n + 255) / 256 : 64);
  if (n == 0) return 0;
  if (wide)
    carry_idle_kernel<uint4><<<dim3(blocks, Bv), 256, 0, (cudaStream_t)stream>>>(
        lengths, reinterpret_cast<const uint4*>(src), reinterpret_cast<uint4*>(dst), n);
  else
    carry_idle_kernel<uint32_t><<<dim3(blocks, Bv), 256, 0, (cudaStream_t)stream>>>(
        lengths, reinterpret_cast<const uint32_t*>(src), reinterpret_cast<uint32_t*>(dst), n);
  LTM_CHECK_LAUNCH("carry_idle");
  return 0;
}

// out[v,s,:] = src[v, idx[v,s], :]
__global__ void __launch_bounds__(256)
gather_rows_kernel(const float4* __restrict__ src, const int32_t* __restrict__ idx, float4* __restrict__ out,
                   int rows_src, int S, int e4) {
  const int s = blockIdx.x, v = blockIdx.y;
  const int row = idx[(size_t)v * S + s];
  for (int c = threadIdx.x; c < e4; c += blockDim.x) {
    float4 val = make_float4(0.f, 0.f, 0.f, 0.f);
    if (row >= 0 && row < rows_src) val = src[((size_t)v * rows_src + row) * e4 + c];
    out[((size_t)v * S + s) * e4 + c] = val;
  }
}

}  // namespace ltm

extern "C" int ltm_consolidate_rect(const float* B_past, const float* xpart, const int32_t* idx,
                                    const uint8_t* new_doc,
                                    const int32_t* seg_ptr0, const int32_t* seg_mem0, const float* g0,
                                    const int32_t* seg_ptr1, const int32_t* seg_mem1, const float* g1,
                                    float* B_new, int Bv, int N, int e, int L, int splits, int S, void* stream) {
  return ltm_consolidate_rect_h(B_past, xpart, idx, new_doc, seg_ptr0, seg_mem0, g0, seg_ptr1, seg_mem1, g1, B_new,
                                nullptr, Bv, N, e, L, splits, S, stream);
}

extern "C" int ltm_consolidate_rect_h(const float* B_past, const float* xpart, const int32_t* idx,
                                      const uint8_t* new_doc,
                                      const int32_t* seg_ptr0, const int32_t* seg_mem0, const float* g0,
                                      const int32_t* seg_ptr1, const int32_t* seg_mem1, const float* g1,
                                      float* B_new, void* B_half, int Bv, int N, int e, int L, int splits, int S,
                                      void* stream) {
  return ltm_consolidate_rect_kv(B_past, xpart, idx, S, new_doc, seg_ptr0, seg_mem0, g0, seg_ptr1, seg_mem1, g1, B_new,
                                 B_half, nullptr, nullptr, nullptr, 0, 0, 0, Bv, N, e, L, splits, S, stream);
}

extern "C" int ltm_consolidate_rect_kv(const float* B_past, const float* xpart, const int32_t* idx, int64_t idx_stride,
                                       const uint8_t* new_doc,
                                       const int32_t* seg_ptr0, const int32_t* seg_mem0, const float* g0,
                                       const int32_t* seg_ptr1, const int32_t* seg_mem1, const float* g1,
                                       float* B_new, void* B_half,
                                       const float* KV_past, float* KV_new, const float* bkv, int ldkv, int jf,
                                       int round_tf32, int Bv, int N, int e, int L, int splits, int S, void* stream) {
  return ltm::consolidate_rect_ragged(B_past, xpart, idx, idx_stride, new_doc, seg_ptr0, seg_mem0, g0, seg_ptr1,
                                      seg_mem1, g1, B_new, B_half, KV_past, KV_new, bkv, ldkv, jf, round_tf32, Bv, N,
                                      e, L, splits, S, nullptr, nullptr, stream);
}

// lengths == NULL: the lock-step kernels.  Otherwise the ragged ones (see Ragged); the tables are the bank's.
int ltm::consolidate_rect_ragged(const float* B_past, const float* xpart, const int32_t* idx, int64_t idx_stride,
                                 const uint8_t* new_doc, const int32_t* seg_ptr0, const int32_t* seg_mem0,
                                 const float* g0, const int32_t* seg_ptr1, const int32_t* seg_mem1, const float* g1,
                                 float* B_new, void* B_half, const float* KV_past, float* KV_new, const float* bkv,
                                 int ldkv, int jf, int round_tf32, int Bv, int N, int e, int L, int splits, int S,
                                 const int32_t* lengths, const int32_t* offs, void* stream) {
  using namespace ltm;
  // round_tf32 == 2: KV_past / KV_new point to fp16 storage [Bv, N, ldkv] (ldkv % 8 == 0)
  const int kv_half = round_tf32 == 2 ? 1 : 0;
  LTM_REQUIRE(B_half == nullptr || (reinterpret_cast<uintptr_t>(B_half) & 7u) == 0, "consolidate_rect: B_half alignment");
  LTM_REQUIRE(xpart && B_new && seg_ptr0 && seg_mem0 && g0, "consolidate_rect: null pointer");
  LTM_REQUIRE(B_past == nullptr || (idx && seg_ptr1 && seg_mem1 && g1),
              "consolidate_rect: update tables / sample indices missing");
  LTM_REQUIRE(B_past != B_new, "consolidate_rect: B_past and B_new must not alias (rows are gathered)");
  LTM_REQUIRE(Bv > 0 && N > 0 && L > 0 && splits > 0 && S > 0 && e > 0 && e % 4 == 0,
              "consolidate_rect: bad shape Bv=%d N=%d e=%d L=%d splits=%d", Bv, N, e, L, splits);
  LTM_REQUIRE(Bv <= 65535, "consolidate_rect: Bv=%d exceeds grid.y", Bv);
  LTM_REQUIRE(aligned16(B_past) && aligned16(xpart) && aligned16(B_new), "consolidate_rect: 16-byte alignment");
  LTM_REQUIRE(idx_stride == 0 || idx_stride >= S, "consolidate_rect: idx_stride=%lld", (long long)idx_stride);
  KvState kv{};
  if (KV_past != nullptr) {
    LTM_REQUIRE(B_past != nullptr && KV_new && bkv && KV_past != KV_new, "consolidate_rect_kv: K|V state needs B_past, "
                "KV_new (distinct from KV_past) and the bias");
    LTM_REQUIRE(ldkv > 0 && ldkv % 4 == 0 && jf >= 0 && jf <= N, "consolidate_rect_kv: bad ldkv=%d / jf=%d", ldkv, jf);
    LTM_REQUIRE(aligned16(KV_past) && aligned16(KV_new) && aligned16(bkv), "consolidate_rect_kv: 16-byte alignment");
    kv.KV_past = reinterpret_cast<const float4*>(KV_past);
    kv.KV_new = reinterpret_cast<float4*>(KV_new);
    kv.bkv = reinterpret_cast<const float4*>(bkv);
    LTM_REQUIRE(!kv_half || ldkv % 8 == 0, "consolidate_rect_kv: fp16 K|V rows need ldkv %% 8 == 0");
    kv.ldkv4 = ldkv / 4; kv.jf = jf; kv.round_tf32 = kv_half ? 0 : round_tf32; kv.half = kv_half;
  }
  const int e4 = e / 4;
  const int threads = e4 >= 256 ? 256 : ((e4 + 31) / 32) * 32;
  // four coefficient rows per CTA once there are plenty of rows: a row is ~10 dependent loads per thread, and four in
  // a row amortise the CTA's launch and tail (measured at 128 videos x 256 bins: consolidate 0.109 -> 0.101 ms alone,
  // the overlapped step 190.2 k -> 195.1 k chunks/s on the same box; 8 rows: no further gain)
  // (num_basis 64 x 1024 videos: 5 % slower with four rows under the overlap -- its rows are longer, 8-10 members each)
  const int rows_per_cta = (N >= 128 && (long long)N * Bv >= 16384) ? 4 : 1;
  dim3 grid((N + rows_per_cta - 1) / rows_per_cta, Bv);
  LTM_REQUIRE((lengths == nullptr) == (offs == nullptr), "consolidate_rect: ragged batches need lengths and offsets");
  const Ragged rg{lengths, offs};
#define LTM_CONSOLIDATE(ROWS, RAGGED)                                                                                 \
  consolidate_rect_kernel<ROWS, RAGGED><<<grid, threads, 0, (cudaStream_t)stream>>>(                                  \
      reinterpret_cast<const float4*>(B_past), reinterpret_cast<const float4*>(xpart), idx, (long long)idx_stride,   \
      new_doc, seg_ptr0, seg_mem0, g0, seg_ptr1, seg_mem1, g1, reinterpret_cast<float4*>(B_new),                     \
      reinterpret_cast<uint2*>(B_half), kv, N, e4, L, splits, S, rg)
  if (rows_per_cta == 4) {
    if (lengths) LTM_CONSOLIDATE(4, true); else LTM_CONSOLIDATE(4, false);
  } else {
    if (lengths) LTM_CONSOLIDATE(1, true); else LTM_CONSOLIDATE(1, false);
  }
#undef LTM_CONSOLIDATE
  LTM_CHECK_LAUNCH("consolidate_rect");
  return 0;
}

extern "C" int ltm_gather_rows(const float* src, const int32_t* idx, float* out, int Bv, int rows_src, int S,
                               int e, void* stream) {
  using namespace ltm;
  LTM_REQUIRE(src && idx && out, "gather_rows: null pointer");
  LTM_REQUIRE(Bv > 0 && Bv <= 65535 && S > 0 && e > 0 && e % 4 == 0, "gather_rows: bad shape");
  LTM_REQUIRE(aligned16(src) && aligned16(out), "gather_rows: 16-byte alignment");
  const int e4 = e / 4;
  const int threads = e4 >= 256 ? 256 : ((e4 + 31) / 32) * 32;
  dim3 grid(S, Bv);
  gather_rows_kernel<<<grid, threads, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<const float4*>(src), idx, reinterpret_cast<float4*>(out), rows_src, S, e4);
  LTM_CHECK_LAUNCH("gather_rows");
  return 0;
}

extern "C" int ltm_fold_sample_columns(const float* GT, int64_t ldg, const int32_t* b_sorted, float* out, int Bv, int N,
                                       int S, int L, int nbins, void* stream) {
  using namespace ltm;
  LTM_REQUIRE(GT && b_sorted && out, "fold_sample_columns: null pointer");
  LTM_REQUIRE(Bv > 0 && Bv <= 65535 && N > 0 && S > 0 && L >= 0 && nbins > 0 && nbins <= 256 && ldg >= S + L,
              "fold_sample_columns: bad shape Bv=%d N=%d S=%d L=%d nbins=%d", Bv, N, S, L, nbins);
  const int rows_per_cta = 8;           // one warp per row
  fold_sample_columns_kernel<<<dim3((N + rows_per_cta - 1) / rows_per_cta, Bv), 256, 8 * nbins * sizeof(float),
                               (cudaStream_t)stream>>>(
      GT, (long long)ldg, b_sorted, out, N, S, L, nbins, rows_per_cta);
  LTM_CHECK_LAUNCH("fold_sample_columns");
  return 0;
}
