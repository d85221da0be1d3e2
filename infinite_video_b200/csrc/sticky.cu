// R6 / G3 / R7 -- sticky memories: density histogram over the 128 sticky bins and inverse-CDF
// re-sampling (long_term_attention_gibbs.py:196-208, long_term_attention.py:220-238).
#include "common.cuh"
#include "rect_hist.cuh"

namespace ltm {

// Standalone op: scores[Bv,H,Q,N] -> hist_part[Bv,H,127]; one CTA per (head, video).  q_tiles > 0: one CTA per
// (head, query tile of 32, video) writing hist_part[Bv, H*q_tiles, 127] -- the layout the fused attention kernels
// produce -- used for num_basis 512, whose tensor-core attention works on two basis halves.
__global__ void __launch_bounds__(256)
sticky_hist_rect_kernel(const float* __restrict__ scores, const int32_t* __restrict__ jb,
                        const float* __restrict__ tb, float* __restrict__ hist_part, int H, int Q, int N,
                        int q_tiles) {
  extern __shared__ float smem[];
  const int h = q_tiles > 0 ? blockIdx.x / q_tiles : blockIdx.x, v = blockIdx.y;
  const int q_lo = q_tiles > 0 ? (blockIdx.x % q_tiles) * 32 : 0;
  const int q_hi = q_tiles > 0 ? min(Q, q_lo + 32) : Q;
  const float* S = scores + ((size_t)(v * H + h) * Q) * N;
  constexpr int RT = 32;
  float* Eb = smem;                       // [RT][130]
  float* Zb = Eb + RT * (EDGES + 1);      // [RT]
  float* mr = Zb + RT;                    // [RT]
  float* part = mr + RT;                  // [128]
  float* accum = part + 128;              // [128]
  for (int i = threadIdx.x; i < 128; i += blockDim.x) accum[i] = 0.f;
  for (int q0 = q_lo; q0 < q_hi; q0 += RT) {
    const int rows = min(RT, q_hi - q0);
    __syncthreads();
    // per-row shift m = max(0, max_i z_i) keeps exp() finite; it cancels in E/Z
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    for (int r = warp; r < rows; r += nw) {
      float m = 0.f;
      for (int i = lane; i < EDGES; i += 32) {
        const int j = jb[i];
        if (j >= 0) m = fmaxf(m, S[(size_t)(q0 + r) * N + j]);
      }
      m = warp_max(m);
      if (lane == 0) mr[r] = m;
    }
    __syncthreads();
    rect_hist_tile([&](int r, int j) { return S[(size_t)(q0 + r) * N + j]; }, mr, rows, jb, tb, Eb, Zb, part);
    __syncthreads();
    for (int i = threadIdx.x; i < EDGES - 2; i += blockDim.x) accum[i] += part[i];
  }
  __syncthreads();
  for (int i = threadIdx.x; i < EDGES - 2; i += blockDim.x)
    hist_part[((size_t)v * gridDim.x + blockIdx.x) * (EDGES - 2) + i] = accum[i];
}

// ------------------------------------------------------------------------------------------------
// Gaussian variant histogram: p_i = sum_r Phi((tb_{i+1}-mu_r)/sd_r) - Phi((tb_i-mu_r)/sd_r), i<128
// (Normal.cdf of torch: 0.5*(1+erf((x-loc)*(1/scale)/sqrt(2)))).  grid (video, part): each CTA sums a
// contiguous share of the R rows (in order) into its own partial histogram -- the re-sampling kernel adds the
// partials in a fixed order -- and thread i evaluates the CDF at EDGE i once per row: the upper edge of
// interval i is the lower edge of interval i+1 (one erff per edge instead of two per interval).
// ------------------------------------------------------------------------------------------------
constexpr int HG_THREADS = 160;              // 129 edges
__global__ void __launch_bounds__(HG_THREADS)
sticky_hist_gauss_kernel(const float* __restrict__ mu, const float* __restrict__ sd,
                         const float* __restrict__ tb, float* __restrict__ hist_part, int R, int parts) {
  __shared__ float phi[2][EDGES + 3];
  const int v = blockIdx.x, pt = blockIdx.y;
  const int i = threadIdx.x;               // edge 0..128 (threads beyond idle), interval 0..127
  const int per = (R + parts - 1) / parts;
  const int r0 = pt * per, r1 = min(R, r0 + per);
  const float edge = (i < EDGES) ? tb[i] : 0.f;
  const float* m = mu + (size_t)v * R;
  const float* s = sd + (size_t)v * R;
  float acc = 0.f;
  for (int r = r0; r < r1; ++r) {
    float* ph = phi[(r - r0) & 1];
    if (i < EDGES) {
      const float inv = __frcp_rn(s[r]);
      ph[i] = 0.5f * (1.f + erff(__fdiv_rn((edge - m[r]) * inv, 1.4142135623730951f)));
    }
    __syncthreads();                       // (the other buffer is rewritten only after the next barrier)
    if (i < EDGES - 1) acc += ph[i + 1] - ph[i];
  }
  if (i < EDGES - 1) hist_part[((size_t)v * parts + pt) * (EDGES - 1) + i] = acc;
}

// ------------------------------------------------------------------------------------------------
// Re-sampling.  One CTA (4 warps) per video.
//   1. p = sum of `parts` partial histograms (fixed order), optionally normalised twice like the
//      reference (p/p.sum() at gibbs:203, then again inside Categorical.__init__).
//   2. CDF exactly as torch's CPU multinomial-with-replacement: sequential fp32 running sum (one
//      thread), divided by the total, last entry forced to 1.
//   3. every thread binary-searches its share of the S fp64 uniforms: first category with cdf >= u.
//   4. optional ascending order of the drawn bins (Gaussian variant sorts ts, gauss:238): counting
//      sort -- bin counts via shared atomics, exclusive warp-shuffle prefix scan, run fill.
// ------------------------------------------------------------------------------------------------
constexpr int MAX_CAT = 128;
constexpr int RS_THREADS = 128;

__device__ __forceinline__ float block_sum_128(float v, float* red) {
  v = warp_sum(v);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  const float t = (red[0] + red[1]) + (red[2] + red[3]);      // fixed order -> reproducible
  __syncthreads();
  return t;
}

// RAGGED: videos with lengths[v] == 0 (idle in a ragged batch) are skipped
template <bool RAGGED>
__global__ void __launch_bounds__(RS_THREADS)
resample_kernel(const float* __restrict__ hist_part, int parts, int ncat, int normalize,
                const double* __restrict__ u, const float* __restrict__ bins,
                const int32_t* __restrict__ bin2basis, int sort,
                float* __restrict__ p_out, int32_t* __restrict__ b_draw, int32_t* __restrict__ b_used,
                float* __restrict__ ts, int32_t* __restrict__ idx, int S, const int32_t* __restrict__ lengths) {
  __shared__ float cdf[MAX_CAT];
  __shared__ int cnt[MAX_CAT];
  __shared__ int start_s[MAX_CAT];
  __shared__ float red[4];
  __shared__ float total_s;
  const int v = blockIdx.x, tid = threadIdx.x;
  if (RAGGED && lengths[v] == 0) return;

  // 1. assemble p
  float a = 0.f;
  if (tid < ncat)
    for (int pt = 0; pt < parts; ++pt) a += hist_part[((size_t)v * parts + pt) * ncat + tid];
  if (normalize) {
    const float tot = block_sum_128(a, red);
    a = __fdiv_rn(a, tot);
    const float tot2 = block_sum_128(tid < ncat ? a : 0.f, red);
    a = __fdiv_rn(a, tot2);
  }
  if (tid < ncat) {
    cdf[tid] = a;
    cnt[tid] = 0;
    if (p_out) p_out[(size_t)v * ncat + tid] = a;
  }
  __syncthreads();

  // 2. sequential fp32 cumulative sum, then normalise by the total (must not be re-associated)
  if (tid == 0) {
    float s = 0.f;
    for (int i = 0; i < ncat; ++i) { s = __fadd_rn(s, cdf[i]); cdf[i] = s; }
    total_s = s;
  }
  __syncthreads();
  if (tid < ncat) cdf[tid] = (tid == ncat - 1) ? 1.0f : __fdiv_rn(cdf[tid], total_s);
  __syncthreads();

  // 3. inverse-CDF search
  for (int s = tid; s < S; s += RS_THREADS) {
    const double us = u[(size_t)v * S + s];
    int left = 0, right = ncat;
    while (right - left > 0) {
      const int mid = left + (right - left) / 2;
      if ((double)cdf[mid] < us) left = mid + 1; else right = mid;
    }
    const int b = min(left, ncat - 1);       // only reachable with NaN/garbage histograms
    if (b_draw) b_draw[(size_t)v * S + s] = b;
    if (sort) {
      atomicAdd(&cnt[b], 1);
    } else {
      if (b_used) b_used[(size_t)v * S + s] = b;
      if (ts) ts[(size_t)v * S + s] = bins[b];
      if (idx) idx[(size_t)v * S + s] = bin2basis ? bin2basis[b] : b;
    }
  }
  if (!sort) return;                         // block-uniform
  __syncthreads();

  // 4. counting sort: exclusive scan of the bin counts by warp 0 (4 bins per lane + warp-shuffle scan)
  if (tid < 32) {
    const int per = (ncat + 31) / 32;        // <= 4
    int local[4] = {0, 0, 0, 0};
    int run = 0;
    for (int t = 0; t < per; ++t) {
      const int i = tid * per + t;
      local[t] = (i < ncat) ? cnt[i] : 0;
      run += local[t];
    }
    int incl = run;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int n = __shfl_up_sync(0xffffffffu, incl, o);
      if (tid >= o) incl += n;
    }
    int start = incl - run;
    for (int t = 0; t < per; ++t) {
      const int i = tid * per + t;
      if (i < ncat) start_s[i] = start;
      start += local[t];
    }
  }
  __syncthreads();
  if (tid < ncat) {
    const float tv = bins[tid];
    const int ix = bin2basis ? bin2basis[tid] : tid;
    const int s0 = start_s[tid], s1 = s0 + cnt[tid];
    for (int s = s0; s < s1; ++s) {
      if (b_used) b_used[(size_t)v * S + s] = tid;
      if (ts) ts[(size_t)v * S + s] = tv;
      if (idx) idx[(size_t)v * S + s] = ix;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Density side-output of the Video-LLaMA copy (gibbs:320-343, consumed by relevant_frames.py): for every
// (video, head, query) row the Gibbs density exp(z(t)) on 3 x 256 points, each segment normalised by its own
// trapezoid integral, the concatenation normalised to sum 1.  One warp per row; out[q, v, h, 768].
// ------------------------------------------------------------------------------------------------
constexpr int DENS_PTS = 768;
__global__ void __launch_bounds__(128)
density_rect_kernel(const float* __restrict__ scores, const int32_t* __restrict__ jd, const float* __restrict__ wd,
                    float* __restrict__ out, int Bv, int H, int Q, int N) {
  const int row = blockIdx.x * 4 + (threadIdx.x >> 5);       // (v*H + h)*Q + q
  const int lane = threadIdx.x & 31;
  if (row >= Bv * H * Q) return;
  const int q = row % Q, vh = row / Q, h = vh % H, v = vh / H;
  const float* S = scores + (size_t)row * N;
  float e[DENS_PTS / 32];
  float m = 0.f;
#pragma unroll
  for (int i = 0; i < DENS_PTS / 32; ++i) {
    const int j = jd[i * 32 + lane];
    e[i] = (j >= 0) ? S[j] : 0.f;
    m = fmaxf(m, e[i]);
  }
  m = warp_max(m);
  float tot = 0.f;
#pragma unroll
  for (int seg = 0; seg < 3; ++seg) {
    float z = 0.f;
#pragma unroll
    for (int i = seg * 8; i < seg * 8 + 8; ++i) {
      e[i] = expf(e[i] - m);
      z += wd[i * 32 + lane] * e[i];
    }
    z = warp_sum(z);
#pragma unroll
    for (int i = seg * 8; i < seg * 8 + 8; ++i) {
      e[i] = e[i] / z;
      tot += e[i];
    }
  }
  tot = warp_sum(tot);
  float* dst = out + (((size_t)q * Bv + v) * H + h) * DENS_PTS;
#pragma unroll
  for (int i = 0; i < DENS_PTS / 32; ++i) dst[i * 32 + lane] = e[i] / tot;
}

// KL regulariser of the Gaussian variant (long_term_attention.py:296-304): per (video, head, query) row
//   kl = 1/2 (var/s0^2 - log(var/s0^2) - 1 [+ (mu - mu0)^2 / s0^2  -- only when mu0 <= 0, as upstream tests `mu_0 > 0`])
__global__ void kl_gauss_kernel(const float* __restrict__ mu, const float* __restrict__ sd, float mu0, float s0sq,
                                int with_mean, float* __restrict__ out, long long n) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float var = sd[i] * sd[i];
  const float r = __fdiv_rn(var, s0sq);
  float kl = r - logf(r) - 1.f;
  if (with_mean) {
    const float dm = mu[i] - mu0;
    kl += __fdiv_rn(dm * dm, s0sq);
  }
  out[i] = 0.5f * kl;
}

}  // namespace ltm

extern "C" int ltm_kl_gauss(const float* mu, const float* sd, float mu_0, float sigma_0, float* out, int64_t n,
                            void* stream) {
  using namespace ltm;
  LTM_REQUIRE(mu && sd && out && n > 0, "kl_gauss: null pointer / empty");
  LTM_REQUIRE(sigma_0 > 0.f, "kl_gauss: sigma_0 must be positive");
  kl_gauss_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(mu, sd, mu_0, sigma_0 * sigma_0,
                                                                               mu_0 > 0.f ? 0 : 1, out, (long long)n);
  LTM_CHECK_LAUNCH("kl_gauss");
  return 0;
}

extern "C" int ltm_density_rect(const float* scores, const int32_t* jd, const float* wd, float* out, int Bv, int H,
                                int Q, int N, void* stream) {
  using namespace ltm;
  LTM_REQUIRE(scores && jd && wd && out, "density_rect: null pointer");
  LTM_REQUIRE(Bv > 0 && H > 0 && Q > 0 && N > 0, "density_rect: bad shape");
  const long long rows = (long long)Bv * H * Q;
  LTM_REQUIRE(rows < (1ll << 31), "density_rect: too many rows");
  density_rect_kernel<<<(unsigned)((rows + 3) / 4), 128, 0, (cudaStream_t)stream>>>(scores, jd, wd, out, Bv, H, Q, N);
  LTM_CHECK_LAUNCH("density_rect");
  return 0;
}

extern "C" int ltm_sticky_hist_rect(const float* scores, const int32_t* jb, const float* tb, float* hist_part,
                                    int Bv, int H, int Q, int N, void* stream) {
  using namespace ltm;
  LTM_REQUIRE(scores && jb && tb && hist_part, "sticky_hist_rect: null pointer");
  LTM_REQUIRE(Bv > 0 && Bv <= 65535 && H > 0 && Q > 0 && N > 0, "sticky_hist_rect: bad shape");
  const size_t smem = sizeof(float) * (32 * (EDGES + 1) + 32 + 32 + 128 + 128);
  dim3 grid(H, Bv);
  sticky_hist_rect_kernel<<<grid, 256, smem, (cudaStream_t)stream>>>(scores, jb, tb, hist_part, H, Q, N, 0);
  LTM_CHECK_LAUNCH("sticky_hist_rect");
  return 0;
}

extern "C" int ltm_sticky_hist_rect_tiles(const float* scores, const int32_t* jb, const float* tb, float* hist_part,
                                          int Bv, int H, int Q, int N, void* stream) {
  using namespace ltm;
  LTM_REQUIRE(scores && jb && tb && hist_part, "sticky_hist_rect_tiles: null pointer");
  LTM_REQUIRE(Bv > 0 && Bv <= 65535 && H > 0 && Q > 0 && N > 0, "sticky_hist_rect_tiles: bad shape");
  const size_t smem = sizeof(float) * (32 * (EDGES + 1) + 32 + 32 + 128 + 128);
  const int q_tiles = (Q + 31) / 32;
  dim3 grid(H * q_tiles, Bv);
  sticky_hist_rect_kernel<<<grid, 256, smem, (cudaStream_t)stream>>>(scores, jb, tb, hist_part, H, Q, N, q_tiles);
  LTM_CHECK_LAUNCH("sticky_hist_rect_tiles");
  return 0;
}

extern "C" int ltm_sticky_hist_gauss(const float* mu, const float* sd, const float* tb, float* hist_part,
                                     int Bv, int R, int parts, void* stream) {
  using namespace ltm;
  LTM_REQUIRE(mu && sd && tb && hist_part, "sticky_hist_gauss: null pointer");
  LTM_REQUIRE(Bv > 0 && Bv <= 2147483647 && R > 0 && parts >= 1 && parts <= 65535 && parts <= R,
              "sticky_hist_gauss: bad shape");
  sticky_hist_gauss_kernel<<<dim3(Bv, parts), HG_THREADS, 0, (cudaStream_t)stream>>>(mu, sd, tb, hist_part, R,
                                                                                       parts);
  LTM_CHECK_LAUNCH("sticky_hist_gauss");
  return 0;
}

extern "C" int ltm_resample(const float* hist_part, int parts, int ncat, int normalize, const double* u,
                            const float* bins, const int32_t* bin2basis, int sort,
                            float* p_out, int32_t* b_draw, int32_t* b_used, float* ts, int32_t* idx,
                            int Bv, int S, void* stream) {
  using namespace ltm;
  LTM_REQUIRE(hist_part && u && bins, "resample: null pointer");
  LTM_REQUIRE(ncat >= 1 && ncat <= MAX_CAT, "resample: ncat=%d out of range [1,%d]", ncat, MAX_CAT);
  LTM_REQUIRE(parts >= 1 && Bv > 0 && S > 0, "resample: bad shape");
  resample_kernel<false><<<Bv, RS_THREADS, 0, (cudaStream_t)stream>>>(hist_part, parts, ncat, normalize, u, bins,
                                                                   bin2basis, sort, p_out, b_draw, b_used, ts, idx, S,
                                                                   nullptr);
  LTM_CHECK_LAUNCH("resample");
  return 0;
}

int ltm::resample_ragged(const float* hist_part, int parts, int ncat, int normalize, const double* u, const float* bins,
                         const int32_t* bin2basis, int sort, float* p_out, int32_t* b_draw, int32_t* b_used, float* ts,
                         int32_t* idx, int Bv, int S, const int32_t* lengths, void* stream) {
  LTM_REQUIRE(hist_part && u && bins && lengths, "resample: null pointer");
  LTM_REQUIRE(ncat >= 1 && ncat <= MAX_CAT, "resample: ncat=%d out of range [1,%d]", ncat, MAX_CAT);
  LTM_REQUIRE(parts >= 1 && Bv > 0 && S > 0, "resample: bad shape");
  resample_kernel<true><<<Bv, RS_THREADS, 0, (cudaStream_t)stream>>>(hist_part, parts, ncat, normalize, u, bins,
                                                                  bin2basis, sort, p_out, b_draw, b_used, ts, idx, S,
                                                                  lengths);
  LTM_CHECK_LAUNCH("resample");
  return 0;
}
