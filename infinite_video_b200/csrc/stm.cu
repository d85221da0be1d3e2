// N1 -- short-term cross-attention of the caller (Qformer.py:224-304) around the tcgen05 GEMMs:
//   scores = (q_h W_k,h / sqrt(d)) enc^T      (the key bias adds a per-row constant: softmax-invariant)
//   P      = softmax(scores + mask)            <- ltm_softmax_rows (this file), in place
//   ctx_h  = (P_h enc) W_v,h^T + b_v,h         (rows of P sum to 1)
//   out    = alpha ctx + (1 - alpha) a_long    <- ltm_blend (this file)
// so that neither K nor V of the 8192 short-term tokens is ever materialised.
#include <cuda_fp16.h>

#include "common.cuh"

namespace ltm {

// fp32 -> fp16 (round to nearest even), 8 elements per thread and step: the chunk tokens as operands of the kind::f16
// short-term attention GEMMs (rounded, where the tensor core would truncate fp32 read as tf32)
__global__ void __launch_bounds__(256)
to_half_kernel(const float4* __restrict__ src, uint4* __restrict__ dst, long long n8) {
  const uint64_t pol = policy_evict_first();
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n8; i += (long long)gridDim.x * blockDim.x) {
    const float4 a = ldg_stream(src + 2 * i, pol), b = ldg_stream(src + 2 * i + 1, pol);
    __half2 h;
    uint4 o;
    h = __floats2half2_rn(a.x, a.y); o.x = *reinterpret_cast<const uint32_t*>(&h);
    h = __floats2half2_rn(a.z, a.w); o.y = *reinterpret_cast<const uint32_t*>(&h);
    h = __floats2half2_rn(b.x, b.y); o.z = *reinterpret_cast<const uint32_t*>(&h);
    h = __floats2half2_rn(b.z, b.w); o.w = *reinterpret_cast<const uint32_t*>(&h);
    dst[i] = o;
  }
}

// fp32 -> two IEEE fp16 terms, x ~ hi + lo (hi = rn(x), lo = rn(x - hi): 22 significant bits while |x| >= 2^-3, an
// absolute floor of 2^-25 below), laid out along K as three segments per row so that a PLAIN kind::f16 GEMM over
// K' = 3K computes the three-term product a_hi b_hi + a_lo b_hi + a_hi b_lo -- fp32-grade like the split-TF32 mode, at the
// fp16 rate:   side 0 (A operand): [hi | lo | hi]     side 1 (B operand): [hi | hi | lo]
__global__ void __launch_bounds__(256)
split_half3_kernel(const float4* __restrict__ src, uint4* __restrict__ dst, long long rows, int k8, int side) {
  const long long total = rows * k8;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / k8;
    const int c = (int)(i - r * k8);
    const float4 a = src[2 * i], b = src[2 * i + 1];
    const float x[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
    uint32_t hi[4], lo[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const __half2 h = __floats2half2_rn(x[2 * j], x[2 * j + 1]);
      const float2 hf = __half22float2(h);
      const __half2 l = __floats2half2_rn(x[2 * j] - hf.x, x[2 * j + 1] - hf.y);
      hi[j] = *reinterpret_cast<const uint32_t*>(&h);
      lo[j] = *reinterpret_cast<const uint32_t*>(&l);
    }
    const uint4 H = make_uint4(hi[0], hi[1], hi[2], hi[3]), Lo = make_uint4(lo[0], lo[1], lo[2], lo[3]);
    uint4* row = dst + r * 3 * k8 + c;
    row[0] = H;
    row[k8] = side == 0 ? Lo : H;
    row[2 * k8] = side == 0 ? H : Lo;
  }
}

__global__ void __launch_bounds__(256)
softmax_rows_kernel(float* __restrict__ S, const float* __restrict__ mask, int n, int rows_per_mask, float scale,
                    __half* __restrict__ P16) {
  __shared__ float red[8];
  const int row = blockIdx.x;
  float4* s4 = reinterpret_cast<float4*>(S + (size_t)row * n);
  const float4* m4 = mask ? reinterpret_cast<const float4*>(mask + (size_t)(row / rows_per_mask) * n) : nullptr;
  const int n4 = n >> 2, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  // pass 1: max
  float mx = -INFINITY;
  for (int i = tid; i < n4; i += 256) {
    float4 v = s4[i];
    v.x *= scale; v.y *= scale; v.z *= scale; v.w *= scale;
    if (m4) { const float4 mm = m4[i]; v.x += mm.x; v.y += mm.y; v.z += mm.z; v.w += mm.w; }
    mx = fmaxf(mx, fmaxf(fmaxf(v.x, v.y), fmaxf(v.z, v.w)));
  }
  mx = warp_max(mx);
  if (lane == 0) red[warp] = mx;
  __syncthreads();
  mx = red[0];
#pragma unroll
  for (int w = 1; w < 8; ++w) mx = fmaxf(mx, red[w]);
  __syncthreads();
  // pass 2: exp + sum (row stays in L1/L2: 32 KB at n = 8192)
  float sum = 0.f;
  for (int i = tid; i < n4; i += 256) {
    float4 v = s4[i];
    v.x *= scale; v.y *= scale; v.z *= scale; v.w *= scale;
    if (m4) { const float4 mm = m4[i]; v.x += mm.x; v.y += mm.y; v.z += mm.z; v.w += mm.w; }
    v.x = expf(v.x - mx); v.y = expf(v.y - mx); v.z = expf(v.z - mx); v.w = expf(v.w - mx);
    sum += (v.x + v.y) + (v.z + v.w);
    s4[i] = v;
  }
  sum = warp_sum(sum);
  if (lane == 0) red[warp] = sum;
  __syncthreads();
  sum = ((red[0] + red[1]) + (red[2] + red[3])) + ((red[4] + red[5]) + (red[6] + red[7]));
  const float inv = 1.0f / sum;
  uint2* p2 = P16 ? reinterpret_cast<uint2*>(P16 + (size_t)row * n) : nullptr;
  for (int i = tid; i < n4; i += 256) {
    float4 v = s4[i];
    v.x *= inv; v.y *= inv; v.z *= inv; v.w *= inv;
    if (p2 != nullptr) {                 // probabilities as fp16 (the A operand of the kind::f16 value GEMM)
      const __half2 lo = __floats2half2_rn(v.x, v.y), hi = __floats2half2_rn(v.z, v.w);
      uint2 pk;
      pk.x = *reinterpret_cast<const uint32_t*>(&lo);
      pk.y = *reinterpret_cast<const uint32_t*>(&hi);
      p2[i] = pk;
    } else {
      s4[i] = v;
    }
  }
}

// Rows of up to 8192 scores with fp16 output: the row lives in registers (8 x 128 bit per thread), so the scores are
// read from HBM once and nothing but the fp16 probabilities is written (the general kernel below re-reads the row twice
// and parks the exponentials in S).  Same arithmetic, same reduction order.
__global__ void __launch_bounds__(256)
softmax_rows_reg_kernel(const float* __restrict__ S, const float* __restrict__ mask, int n, int rows_per_mask,
                        float scale, __half* __restrict__ P16) {
  constexpr int ITEMS = 8;
  __shared__ float red[8];
  const int row = blockIdx.x;
  const float4* s4 = reinterpret_cast<const float4*>(S + (size_t)row * n);
  const float4* m4 = mask ? reinterpret_cast<const float4*>(mask + (size_t)(row / rows_per_mask) * n) : nullptr;
  const int n4 = n >> 2, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  float4 v[ITEMS];
#pragma unroll
  for (int k = 0; k < ITEMS; ++k) {
    const int i = tid + 256 * k;
    v[k] = make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
    if (i < n4) {
      asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                   : "=f"(v[k].x), "=f"(v[k].y), "=f"(v[k].z), "=f"(v[k].w) : "l"(s4 + i));
    }
  }
  float mx = -INFINITY;
#pragma unroll
  for (int k = 0; k < ITEMS; ++k) {
    const int i = tid + 256 * k;
    if (i < n4) {
      v[k].x *= scale; v[k].y *= scale; v[k].z *= scale; v[k].w *= scale;
      if (m4) { const float4 mm = m4[i]; v[k].x += mm.x; v[k].y += mm.y; v[k].z += mm.z; v[k].w += mm.w; }
      mx = fmaxf(mx, fmaxf(fmaxf(v[k].x, v[k].y), fmaxf(v[k].z, v[k].w)));
    }
  }
  mx = warp_max(mx);
  if (lane == 0) red[warp] = mx;
  __syncthreads();
  mx = red[0];
#pragma unroll
  for (int w = 1; w < 8; ++w) mx = fmaxf(mx, red[w]);
  __syncthreads();
  float sum = 0.f;
#pragma unroll
  for (int k = 0; k < ITEMS; ++k) {
    if (tid + 256 * k < n4) {
      v[k].x = expf(v[k].x - mx); v[k].y = expf(v[k].y - mx); v[k].z = expf(v[k].z - mx); v[k].w = expf(v[k].w - mx);
      sum += (v[k].x + v[k].y) + (v[k].z + v[k].w);
    }
  }
  sum = warp_sum(sum);
  if (lane == 0) red[warp] = sum;
  __syncthreads();
  sum = ((red[0] + red[1]) + (red[2] + red[3])) + ((red[4] + red[5]) + (red[6] + red[7]));
  const float inv = 1.0f / sum;
  uint2* p2 = reinterpret_cast<uint2*>(P16 + (size_t)row * n);
#pragma unroll
  for (int k = 0; k < ITEMS; ++k) {
    const int i = tid + 256 * k;
    if (i < n4) {
      const __half2 lo = __floats2half2_rn(v[k].x * inv, v[k].y * inv), hi = __floats2half2_rn(v[k].z * inv, v[k].w * inv);
      uint2 pk;
      pk.x = *reinterpret_cast<const uint32_t*>(&lo);
      pk.y = *reinterpret_cast<const uint32_t*>(&hi);
      p2[i] = pk;
    }
  }
}

// Columns 4i .. 4i+3 of a score row of n valid columns, scaled and masked; -inf past n (adds nothing to the max and
// exp() = +0 to the sum).  Columns >= n of S and of the mask are not read.  With a mask, s * scale + m is one fused
// multiply-add (one rounding), as the lock-step kernels compile `v *= scale; v += mm`.
__device__ __forceinline__ float score_len(float s, const float* __restrict__ m, int c, float scale) {
  return m ? __fmaf_rn(s, scale, __ldg(m + c)) : s * scale;
}
__device__ __forceinline__ float4 score4_len(const float* __restrict__ s, const float* __restrict__ m, int i, int n,
                                             float scale) {
  const int c = 4 * i;
  float4 v;
  if (c + 4 <= n) {
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(s + c));
    v.x = score_len(v.x, m, c, scale);
    v.y = score_len(v.y, m, c + 1, scale);
    v.z = score_len(v.z, m, c + 2, scale);
    v.w = score_len(v.w, m, c + 3, scale);
  } else {
    v.x = score_len(__ldg(s + c), m, c, scale);
    v.y = c + 1 < n ? score_len(__ldg(s + c + 1), m, c + 1, scale) : -INFINITY;
    v.z = c + 2 < n ? score_len(__ldg(s + c + 2), m, c + 2, scale) : -INFINITY;
    v.w = c + 3 < n ? score_len(__ldg(s + c + 3), m, c + 3, scale) : -INFINITY;
  }
  return v;
}

__device__ __forceinline__ uint2 half4_scaled(const float4& w, float inv) {
  const __half2 lo = __floats2half2_rn(w.x * inv, w.y * inv), hi = __floats2half2_rn(w.z * inv, w.w * inv);
  return make_uint2(*reinterpret_cast<const uint32_t*>(&lo), *reinterpret_cast<const uint32_t*>(&hi));
}

// Row softmax of a ragged batch with fp16 output: row r belongs to video r / rows_per_len and spans that video's first
// n = n_len[video] columns.  The arithmetic (scale and mask in one FFMA, score4_len) and the reduction order are
// those of softmax_rows_reg_kernel / softmax_rows_kernel on a row of n columns, so a row whose n is a multiple of 4
// gets the same bits, with or without a mask; P columns
// [n, roundup64(n)) are written as +0 (the value GEMM reads whole 64-column k-blocks), nothing beyond.  Rows with
// n = 0 are not touched.  REG: the row (<= 8192 columns) stays in registers; otherwise S is read three times.
template <bool REG>
__global__ void __launch_bounds__(256)
softmax_rows_len_kernel(const float* __restrict__ S, const float* __restrict__ mask, const int32_t* __restrict__ n_len,
                        __half* __restrict__ P16, long long ld, long long mask_ld, int rows_per_len, float scale) {
  constexpr int ITEMS = 8;
  __shared__ float red[8];
  const int row = blockIdx.x, vid = row / rows_per_len;
  const int n = __ldg(n_len + vid);
  if (n <= 0) return;
  const float* s = S + (size_t)row * ld;
  const float* m = mask ? mask + (size_t)vid * mask_ld : nullptr;
  const int nq = (n + 3) >> 2, n64q = ((n + 63) & ~63) >> 2, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  float4 v[REG ? ITEMS : 1];
  float mx = -INFINITY;
  if (REG) {
#pragma unroll
    for (int k = 0; k < ITEMS; ++k) {
      const int i = tid + 256 * k;
      v[k] = make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
      if (i < nq) {
        v[k] = score4_len(s, m, i, n, scale);
        mx = fmaxf(mx, fmaxf(fmaxf(v[k].x, v[k].y), fmaxf(v[k].z, v[k].w)));
      }
    }
  } else {
    for (int i = tid; i < nq; i += 256) {
      const float4 w = score4_len(s, m, i, n, scale);
      mx = fmaxf(mx, fmaxf(fmaxf(w.x, w.y), fmaxf(w.z, w.w)));
    }
  }
  mx = warp_max(mx);
  if (lane == 0) red[warp] = mx;
  __syncthreads();
  mx = red[0];
#pragma unroll
  for (int w = 1; w < 8; ++w) mx = fmaxf(mx, red[w]);
  __syncthreads();
  float sum = 0.f;
  if (REG) {
#pragma unroll
    for (int k = 0; k < ITEMS; ++k) {
      if (tid + 256 * k < nq) {
        v[k].x = expf(v[k].x - mx); v[k].y = expf(v[k].y - mx); v[k].z = expf(v[k].z - mx); v[k].w = expf(v[k].w - mx);
        sum += (v[k].x + v[k].y) + (v[k].z + v[k].w);
      }
    }
  } else {
    for (int i = tid; i < nq; i += 256) {
      float4 w = score4_len(s, m, i, n, scale);
      w.x = expf(w.x - mx); w.y = expf(w.y - mx); w.z = expf(w.z - mx); w.w = expf(w.w - mx);
      sum += (w.x + w.y) + (w.z + w.w);
    }
  }
  sum = warp_sum(sum);
  if (lane == 0) red[warp] = sum;
  __syncthreads();
  sum = ((red[0] + red[1]) + (red[2] + red[3])) + ((red[4] + red[5]) + (red[6] + red[7]));
  const float inv = 1.0f / sum;
  uint2* p2 = reinterpret_cast<uint2*>(P16 + (size_t)row * ld);
  if (REG) {
#pragma unroll
    for (int k = 0; k < ITEMS; ++k) {
      const int i = tid + 256 * k;
      if (i < n64q) p2[i] = i < nq ? half4_scaled(v[k], inv) : make_uint2(0u, 0u);   // then the zero tail
    }
  } else {
    for (int i = tid; i < n64q; i += 256) {
      uint2 pk = make_uint2(0u, 0u);
      if (i < nq) {
        float4 w = score4_len(s, m, i, n, scale);
        w.x = expf(w.x - mx); w.y = expf(w.y - mx); w.z = expf(w.z - mx); w.w = expf(w.w - mx);
        pk = half4_scaled(w, inv);
      }
      p2[i] = pk;
    }
  }
}

__global__ void blend_kernel(const float4* __restrict__ a, const float4* __restrict__ b, float alpha,
                             float4* __restrict__ out, long long n4) {
  const float beta = 1.0f - alpha;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    const float4 x = a[i], y = b[i];
    out[i] = make_float4(alpha * x.x + beta * y.x, alpha * x.y + beta * y.y, alpha * x.z + beta * y.z,
                         alpha * x.w + beta * y.w);
  }
}

}  // namespace ltm

extern "C" int ltm_softmax_rows(float* S, const float* mask, int rows, int n, int rows_per_mask, float scale,
                                void* stream) {
  using namespace ltm;
  LTM_REQUIRE(S != nullptr, "softmax_rows: null pointer");
  LTM_REQUIRE(rows > 0 && n > 0 && n % 4 == 0, "softmax_rows: bad shape rows=%d n=%d (n %% 4 == 0)", rows, n);
  LTM_REQUIRE(mask == nullptr || rows_per_mask > 0, "softmax_rows: rows_per_mask must be positive");
  LTM_REQUIRE(aligned16(S) && aligned16(mask), "softmax_rows: 16-byte alignment");
  softmax_rows_kernel<<<rows, 256, 0, (cudaStream_t)stream>>>(S, mask, n, rows_per_mask > 0 ? rows_per_mask : 1, scale,
                                                              nullptr);
  LTM_CHECK_LAUNCH("softmax_rows");
  return 0;
}

extern "C" int ltm_softmax_rows_h(float* S, const float* mask, void* P16, int rows, int n, int rows_per_mask,
                                  float scale, void* stream) {
  using namespace ltm;
  LTM_REQUIRE(S != nullptr && P16 != nullptr, "softmax_rows_h: null pointer");
  LTM_REQUIRE(rows > 0 && n > 0 && n % 4 == 0, "softmax_rows_h: bad shape rows=%d n=%d (n %% 4 == 0)", rows, n);
  LTM_REQUIRE(mask == nullptr || rows_per_mask > 0, "softmax_rows_h: rows_per_mask must be positive");
  LTM_REQUIRE(aligned16(S) && aligned16(mask) && (reinterpret_cast<uintptr_t>(P16) & 7u) == 0, "softmax_rows_h: alignment");
  if (n <= 8192)   // the row fits the registers of one CTA: one pass over HBM (S is left untouched)
    softmax_rows_reg_kernel<<<rows, 256, 0, (cudaStream_t)stream>>>(S, mask, n, rows_per_mask > 0 ? rows_per_mask : 1,
                                                                    scale, reinterpret_cast<__half*>(P16));
  else
    softmax_rows_kernel<<<rows, 256, 0, (cudaStream_t)stream>>>(S, mask, n, rows_per_mask > 0 ? rows_per_mask : 1, scale,
                                                                reinterpret_cast<__half*>(P16));
  LTM_CHECK_LAUNCH("softmax_rows_h");
  return 0;
}

extern "C" int ltm_softmax_rows_h_len(const float* S, const float* mask, void* P16, const int32_t* n_len, int rows, int ld,
                                      int mask_ld, int rows_per_len, float scale, void* stream) {
  using namespace ltm;
  LTM_REQUIRE(S != nullptr && P16 != nullptr && n_len != nullptr, "softmax_rows_h_len: null pointer");
  LTM_REQUIRE(rows > 0 && ld > 0 && ld % 64 == 0 && rows_per_len > 0 && rows % rows_per_len == 0,
              "softmax_rows_h_len: bad shape rows=%d ld=%d rows_per_len=%d (ld %% 64 == 0, rows %% rows_per_len == 0)",
              rows, ld, rows_per_len);
  LTM_REQUIRE(mask == nullptr || mask_ld > 0, "softmax_rows_h_len: mask_ld must be positive");
  LTM_REQUIRE(aligned16(S) && aligned16(P16), "softmax_rows_h_len: 16-byte alignment");
  if (ld <= 8192)   // every row fits the registers of one CTA
    softmax_rows_len_kernel<true><<<rows, 256, 0, (cudaStream_t)stream>>>(
        S, mask, n_len, reinterpret_cast<__half*>(P16), ld, mask_ld, rows_per_len, scale);
  else
    softmax_rows_len_kernel<false><<<rows, 256, 0, (cudaStream_t)stream>>>(
        S, mask, n_len, reinterpret_cast<__half*>(P16), ld, mask_ld, rows_per_len, scale);
  LTM_CHECK_LAUNCH("softmax_rows_h_len");
  return 0;
}

extern "C" int ltm_to_half(const float* src, void* dst, int64_t n, void* stream) {
  using namespace ltm;
  LTM_REQUIRE(src && dst, "to_half: null pointer");
  LTM_REQUIRE(n > 0 && n % 8 == 0 && aligned16(src) && aligned16(dst), "to_half: n %% 8 == 0 and 16-byte alignment");
  const long long n8 = n / 8;
  const int blocks = (int)((n8 + 255) / 256 < 148 * 16 ? (n8 + 255) / 256 : 148 * 16);
  to_half_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const float4*>(src),
                                                           reinterpret_cast<uint4*>(dst), n8);
  LTM_CHECK_LAUNCH("to_half");
  return 0;
}

extern "C" int ltm_split_half3(const float* src, void* dst, int64_t rows, int K, int side, void* stream) {
  using namespace ltm;
  LTM_REQUIRE(src && dst, "split_half3: null pointer");
  LTM_REQUIRE(rows > 0 && K > 0 && K % 8 == 0 && (side == 0 || side == 1) && aligned16(src) && aligned16(dst),
              "split_half3: rows=%lld K=%d (K %% 8 == 0), side 0 / 1, 16-byte alignment", (long long)rows, K);
  const long long total = rows * (K / 8);
  const int blocks = (int)((total + 255) / 256 < 148 * 16 ? (total + 255) / 256 : 148 * 16);
  split_half3_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const float4*>(src),
                                                               reinterpret_cast<uint4*>(dst), rows, K / 8, side);
  LTM_CHECK_LAUNCH("split_half3");
  return 0;
}

extern "C" int ltm_blend(const float* a, const float* b, float alpha, float* out, int64_t n, void* stream) {
  using namespace ltm;
  LTM_REQUIRE(a && b && out, "blend: null pointer");
  LTM_REQUIRE(n > 0 && n % 4 == 0, "blend: n=%lld must be a positive multiple of 4", (long long)n);
  LTM_REQUIRE(aligned16(a) && aligned16(b) && aligned16(out), "blend: 16-byte alignment");
  const long long n4 = n / 4;
  const int blocks = (int)((n4 + 255) / 256 < 148 * 8 ? (n4 + 255) / 256 : 148 * 8);
  blend_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const float4*>(a),
                                                          reinterpret_cast<const float4*>(b), alpha,
                                                          reinterpret_cast<float4*>(out), n4);
  LTM_CHECK_LAUNCH("blend");
  return 0;
}
