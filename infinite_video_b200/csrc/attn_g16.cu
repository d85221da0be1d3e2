// Continuous attention of variant G (Gaussian RBF bases) on the tensor cores (G4, long_term_attention.py:286-325).
//
// Same pipeline and work decomposition as the fp16 path of attn_tc.cu (read that file's header first): persistent CTAs
// walk the work items (query tile, head, video); per item one thread issues  S^T = K_h q_h^T  and  D = V_h^T r  as
// kind::f16 UMMAs with fp32 accumulation in TMEM while eight compute warps turn the scores into the weights r.  What
// differs:
//
//   * precision.  softmax(20 S) amplifies score errors twenty-fold and the weights r_j reach ~80 with the coefficients
//     of an ill-conditioned ridge regression behind V, so single-pass fp16 / tf32 products are not enough (measured:
//     1.1e-3 on the context).  Every operand comes as TWO fp16 terms, x ~ hi + lo (22 significant bits): K|V from the
//     projection GEMM's epilogue (ltm_gemm C_lo), q / sqrt(d) and r split by the CTA, and each contraction is issued as
//     the three products  hi.hi + lo.hi + hi.lo  accumulating into the same TMEM columns -- fp32-grade results at the
//     fp16 tensor rate (the "fp16x2" scheme of ltm_split_half3, here without any duplicated operand in memory).
//   * the weights.  a = softmax_j(20 S)  ->  mu = a.mu_b,  E[t^2] = a.(mu_b^2 + sigma_b^2),  var = E[t^2] - mu^2
//     (fp64 sums, rounded to fp32 before the cancelling subtraction exactly like attn_fast.cu)  ->  canonical-parameter
//     round trip of the reference (gauss:308-310)  ->  r_j = N(mu; mu_b_j, sigma_b_j^2 + var).  The column statistics
//     over the 256 basis rows are warp-transposing shuffle reductions (31 shuffles for 32 columns) + one shared-memory
//     hop across the warps.
//   * no normaliser rows, no histogram: ctx = r V directly; mu and sd go out for the erf histogram kernel.
//
// Shared memory per CTA at num_basis 256: K hi/lo 64 KB + V hi/lo 64 KB + r^T hi/lo 32 KB + q hi/lo 8 KB.
#include <cuda_fp16.h>

#include <cudaTypedefs.h>

#include "tcgen05.cuh"

namespace ltm {
namespace g16 {

constexpr int DH = 64;
constexpr int QT = 32;
constexpr int THREADS = 320;             // 8 compute warps (TMEM lane quarter = warp % 4) + 2 issuing warps
constexpr int MAX_REGS = 168;            // three 32-column fp64 reductions live next to the 32 scores of a thread
constexpr int TMEM_COLS = 128;           // S^T: NB/128 x 32 columns at 0; D: 2 x 32 columns at 64 (one per issuer)

struct Params {
  const float* q;        // [Bv,Q,D]
  const float* bmu;      // [NB] basis centres
  const float* bsig;     // [NB] basis widths
  float* ctx;            // [Bv,Q,D]
  float* mu_out;         // [Bv,H*Q]
  float* sd_out;         // [Bv,H*Q]
  int Q, H;
};

template <int NB>
struct Lay {
  static constexpr int SLAB = NB * 128;              // NB rows x 64 halves
  static constexpr int KH_OFF = 0, KL_OFF = SLAB;    // K_h[j][64 d] hi | lo          (K-major rows = j)
  static constexpr int VH_OFF = 2 * SLAB, VL_OFF = 3 * SLAB;   // V_h[j][64 d] hi | lo (MN-major rows = j)
  static constexpr int R_BYTES = ((NB + 63) / 64) * 4096;     // r^T: [NB/64 k-blocks][32 q][64 j]
  static constexpr int RH_OFF = 4 * SLAB, RL_OFF = RH_OFF + R_BYTES;
  static constexpr int QH_OFF = RL_OFF + R_BYTES, QL_OFF = QH_OFF + 4096;      // q tile hi | lo: [32 q][64 d]
  static constexpr int MISC_OFF = QL_OFF + 4096;
  // wmax[8][32] floats | psum[3][8][32] doubles | murt[32] varrt[32] floats
  static constexpr int MISC_BYTES = 8 * 32 * 4 + 3 * 8 * 32 * 8 + 2 * 32 * 4;
  static constexpr int BYTES = MISC_OFF + MISC_BYTES + 64 + 1024;   // + 6 barriers, TMEM slot, alignment slack
  // the M = 128 instructions read one slab past a 64-row operand and the second MN atom of a value operand lies one
  // slab behind it: both stay inside this allocation (K_lo -> V_hi, V_lo -> the r^T tiles), finite or not those rows
  // only reach accumulator lanes nobody reads
  static_assert(2 * R_BYTES >= SLAB || NB == 64, "second MN atom of V_lo must stay inside the r^T tiles");
};

__device__ __forceinline__ void cw_sync() { asm volatile("bar.sync 1, 256;" ::: "memory"); }   // the 8 compute warps

struct QRegs { float4 a, b; };
__device__ __forceinline__ QRegs load_q(const float* qbase, int rows, int D, int tid) {
  const int qq = tid >> 3, dch = tid & 7;                          // 8 consecutive d per thread
  QRegs r;
  r.a = make_float4(0.f, 0.f, 0.f, 0.f);
  r.b = r.a;
  if (qq < rows) {
    const float4* src = reinterpret_cast<const float4*>(qbase + (size_t)qq * D + dch * 8);
    r.a = __ldg(src);
    r.b = __ldg(src + 1);
  }
  return r;
}
__device__ __forceinline__ void split2(float x, float y, uint32_t& hi, uint32_t& lo) {
  const __half2 h = __floats2half2_rn(x, y);
  const float2 hf = __half22float2(h);
  const __half2 l = __floats2half2_rn(x - hf.x, y - hf.y);
  hi = *reinterpret_cast<const uint32_t*>(&h);
  lo = *reinterpret_cast<const uint32_t*>(&l);
}
// q / sqrt(d) (gauss:286; a power of two, exact) as hi + lo fp16 tiles in the K-major SWIZZLE_128B layout: row q = 64
// halves = 128 B, 16-byte chunk (d >> 3) at position (d >> 3) ^ (q & 7)
__device__ __forceinline__ void store_q_tiles(uint8_t* qh, uint8_t* ql, const QRegs& r, int tid) {
  const int qq = tid >> 3, dch = tid & 7;
  const float sc = 0.125f;
  uint4 H, L;
  split2(r.a.x * sc, r.a.y * sc, H.x, L.x);
  split2(r.a.z * sc, r.a.w * sc, H.y, L.y);
  split2(r.b.x * sc, r.b.y * sc, H.z, L.z);
  split2(r.b.z * sc, r.b.w * sc, H.w, L.w);
  const int off = qq * 128 + ((dch ^ (qq & 7)) << 4);
  *reinterpret_cast<uint4*>(qh + off) = H;
  *reinterpret_cast<uint4*>(ql + off) = L;
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

// Column statistics over the lanes of a warp: every lane holds 32 values (one per column); afterwards lane c holds the
// reduction of column c over the 32 lanes.  16 + 8 + 4 + 2 + 1 = 31 exchanges instead of 32 x 5.
template <typename T, typename Op>
__device__ __forceinline__ T warp_transpose_reduce(T (&v)[32], int lane, Op op) {
#pragma unroll
  for (int half = 16; half >= 1; half >>= 1) {
    const bool up = (lane & half) != 0;
#pragma unroll
    for (int i = 0; i < half; ++i) {
      const T send = up ? v[i] : v[i + half];
      const T recv = __shfl_xor_sync(0xffffffffu, send, half);
      v[i] = op(up ? v[i + half] : v[i], recv);
    }
  }
  return v[0];
}

template <int NB>
__global__ void __maxnreg__(MAX_REGS)
cont_attn_g16_kernel(const __grid_constant__ CUtensorMap mapKh, const __grid_constant__ CUtensorMap mapKl,
                     const __grid_constant__ CUtensorMap mapVh, const __grid_constant__ CUtensorMap mapVl,
                     const Params p, const int q_tiles, const int total) {
  static_assert(NB == 64 || NB == 128 || NB == 256, "the tensor-core path covers num_basis 64 / 128 / 256");
  using L_ = Lay<NB>;
  constexpr int HALVES = (NB + 127) / 128;   // score MMAs (M = 128 each)
  constexpr int JWARPS = NB / 32;            // compute warps that own a basis
  extern __shared__ uint8_t smem_raw[];
  const uint32_t sbase = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* sm = smem_raw + (sbase - smem_u32(smem_raw));
  float* wmax = reinterpret_cast<float*>(sm + L_::MISC_OFF);                 // [8][32]
  double* psum = reinterpret_cast<double*>(sm + L_::MISC_OFF + 8 * 32 * 4);  // [3][8][32]
  float* murt = reinterpret_cast<float*>(sm + L_::MISC_OFF + 8 * 32 * 4 + 3 * 8 * 32 * 8);
  float* varrt = murt + 32;
  const uint32_t bars = sbase + L_::MISC_OFF + L_::MISC_BYTES;
  const uint32_t bar_k = bars, bar_v = bars + 8, bar_s = bars + 16, bar_pv = bars + 24, bar_q = bars + 32,
                 bar_r = bars + 40;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(sm + L_::MISC_OFF + L_::MISC_BYTES + 48);

  const int Q = p.Q, H = p.H, D = H * DH;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t sKh = sbase + L_::KH_OFF, sKl = sbase + L_::KL_OFF, sVh = sbase + L_::VH_OFF, sVl = sbase + L_::VL_OFF;
  const uint32_t sRh = sbase + L_::RH_OFF, sRl = sbase + L_::RL_OFF, sQh = sbase + L_::QH_OFF, sQl = sbase + L_::QL_OFF;
  const int nvid = total / (H * q_tiles);
  // videos are walked last-to-first: the projection that ran just before wrote K|V first-to-last
  auto decode = [&](int w, int& qt, int& h, int& v) {
    h = w % H;
    qt = (w / H) % q_tiles;
    v = nvid - 1 - w / (H * q_tiles);
  };
  const int w0 = blockIdx.x, wstride = gridDim.x;

  if (warp == 8) {
    if (lane == 0) {
      asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&mapKh)) : "memory");
      asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&mapKl)) : "memory");
      asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&mapVh)) : "memory");
      asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&mapVl)) : "memory");
      mbar_init(bar_k, 1);
      mbar_init(bar_v, 1);
      mbar_init(bar_s, 1);
      mbar_init(bar_pv, 2);                            // one commit per issuing warp
      mbar_init(bar_q, 256);
      mbar_init(bar_r, 256);
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
      int qt, h, v;
      decode(w0, qt, h, v);
      mbar_arrive_expect_tx(bar_k, 2 * L_::SLAB);
      tma_load_2d(&mapKh, sKh, bar_k, h * DH, v * NB);
      tma_load_2d(&mapKl, sKl, bar_k, h * DH, v * NB);
      mbar_arrive_expect_tx(bar_v, 2 * L_::SLAB);
      tma_load_2d(&mapVh, sVh, bar_v, h * DH, v * NB);
      tma_load_2d(&mapVl, sVl, bar_v, h * DH, v * NB);
    }
    __syncwarp();
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                 "r"((uint32_t)TMEM_COLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tcgen05_fence_before();
  __syncthreads();                       // barriers initialised, TMEM allocated
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  // instruction descriptors: D=f32 [4,6)=1, A=f16 [7,10)=0, B=f16 [10,13)=0, a_major bit 15 (1 = MN-major),
  // N>>3 [17,23), M>>4 [24,29)
  constexpr uint32_t IDESC_S = (1u << 4) | ((uint32_t)(QT >> 3) << 17) | ((128u >> 4) << 24);
  constexpr uint32_t IDESC_PV = IDESC_S | (1u << 15);

  // PV products of the k-steps [k0, k1): hi.hi + lo.hi + hi.lo into one accumulator
  auto issue_pv = [&](uint32_t dcol, int k0, int k1) {
    const uint64_t dVh = umma_desc(sVh, L_::SLAB, 1024, 2u), dVl = umma_desc(sVl, L_::SLAB, 1024, 2u);
    const uint64_t dRh = umma_desc(sRh, 16, 1024, 2u), dRl = umma_desc(sRl, 16, 1024, 2u);
    const uint32_t hiw = (uint32_t)(dVh >> 32), rhiw = (uint32_t)(dRh >> 32);
    const uint32_t va[3] = {(uint32_t)dVh, (uint32_t)dVl, (uint32_t)dVh};
    const uint32_t rb[3] = {(uint32_t)dRh, (uint32_t)dRh, (uint32_t)dRl};
#pragma unroll
    for (int t = 0; t < 3; ++t) {
      for (int ks = k0; ks < k1; ++ks)
        tcgen05_mma_f16(tmem_base + dcol, va[t] + (uint32_t)((ks * 2048) >> 4), hiw,
                        rb[t] + (uint32_t)(((ks >> 2) * 4096 + (ks & 3) * 32) >> 4), rhiw, IDESC_PV,
                        (t != 0 || ks != k0) ? 1u : 0u);
    }
  };

  if (warp == 8) {
    // ------------------------------------------------------------------ TMA + MMA issue (one lane)
    if (lane == 0) {
      const uint64_t dKh = umma_desc(sKh, 16, 1024, 2u), dKl = umma_desc(sKl, 16, 1024, 2u);
      const uint64_t dQh = umma_desc(sQh, 16, 1024, 2u), dQl = umma_desc(sQl, 16, 1024, 2u);
      const uint32_t khiw = (uint32_t)(dKh >> 32);
      const uint32_t ka[3] = {(uint32_t)dKh, (uint32_t)dKl, (uint32_t)dKh};
      const uint32_t qb[3] = {(uint32_t)dQh, (uint32_t)dQh, (uint32_t)dQl};
      auto issue_scores = [&](uint32_t ph) {           // S^T of the item whose K tiles / q tiles carry parity ph
        mbar_wait(bar_q, ph);                          // q tiles written, S read out of TMEM
        mbar_wait(bar_k, ph);
        tcgen05_fence_after();
#pragma unroll
        for (int hf = 0; hf < HALVES; ++hf) {
#pragma unroll
          for (int t = 0; t < 3; ++t) {
#pragma unroll
            for (int ks = 0; ks < DH / 16; ++ks)
              tcgen05_mma_f16(tmem_base + hf * QT, ka[t] + (uint32_t)((hf * (128 * 128) + ks * 32) >> 4), khiw,
                              qb[t] + (uint32_t)((ks * 32) >> 4), khiw, IDESC_S, (t != 0 || ks != 0) ? 1u : 0u);
          }
        }
        tcgen05_commit(bar_s);
      };
      uint32_t it = 0;
      issue_scores(0u);
      for (int w = w0; w < total; w += wstride, ++it) {
        const uint32_t ph = it & 1u;
        const int wn = w + wstride;
        int qtn = 0, hn = 0, vn = 0;
        if (wn < total) decode(wn, qtn, hn, vn);
        mbar_wait(bar_s, ph);                          // the K buffers have been read
        if (wn < total) {
          mbar_arrive_expect_tx(bar_k, 2 * L_::SLAB);
          tma_load_2d(&mapKh, sKh, bar_k, hn * DH, vn * NB);
          tma_load_2d(&mapKl, sKl, bar_k, hn * DH, vn * NB);
        }
        mbar_wait(bar_r, ph);                          // r^T written, D free
        mbar_wait(bar_v, ph);
        tcgen05_fence_after();
        issue_pv(64u, 0, NB / 32);                     // first half of the basis range into D0 (warp 9: second half, D1)
        tcgen05_commit(bar_pv);
        if (wn < total) issue_scores(ph ^ 1u);
        mbar_wait(bar_pv, ph);                         // the V buffers (and r^T) have been read
        if (wn < total) {
          mbar_arrive_expect_tx(bar_v, 2 * L_::SLAB);
          tma_load_2d(&mapVh, sVh, bar_v, hn * DH, vn * NB);
          tma_load_2d(&mapVl, sVl, bar_v, hn * DH, vn * NB);
        }
      }
    }
    __syncwarp();
  } else if (warp == 9) {
    // ------------------------------------------------------------------ second MMA issuer (one lane)
    if (lane == 0) {
      uint32_t it = 0;
      for (int w = w0; w < total; w += wstride, ++it) {
        const uint32_t ph = it & 1u;
        mbar_wait(bar_r, ph);
        mbar_wait(bar_v, ph);
        tcgen05_fence_after();
        issue_pv(96u, NB / 32, NB / 16);
        tcgen05_commit(bar_pv);
      }
    }
    __syncwarp();
  } else {
    // ------------------------------------------------------------------ compute warps
    const bool active = warp < JWARPS;
    const int j = (warp >> 2) * 128 + (warp & 3) * 32 + lane;      // this thread's basis in the weight phase
    const int quarter = warp & 3, chalf = warp >> 2;
    const float bm = active ? __ldg(p.bmu + j) : 0.f;
    const float bs = active ? __ldg(p.bsig + j) : 1.f;
    const float c2 = __fadd_rn(__fmul_rn(bm, bm), __fmul_rn(bs, bs));     // mu_b^2 + sigma_b^2 (gauss:291)
    const float bs2 = __fmul_rn(bs, bs);
    {
      int qt, h, v;
      decode(w0, qt, h, v);
      const QRegs qr = load_q(p.q + ((size_t)v * Q + qt * QT) * D + h * DH, min(QT, Q - qt * QT), D, tid);
      store_q_tiles(sm + L_::QH_OFF, sm + L_::QL_OFF, qr, tid);
      mbar_arrive(bar_q);
    }
    QRegs qnext;                                       // queries of item it + 1, fetched during item it - 1
    qnext.a = make_float4(0.f, 0.f, 0.f, 0.f);
    qnext.b = qnext.a;
    if (w0 + wstride < total) {
      int qtn, hn, vn;
      decode(w0 + wstride, qtn, hn, vn);
      qnext = load_q(p.q + ((size_t)vn * Q + qtn * QT) * D + hn * DH, min(QT, Q - qtn * QT), D, tid);
    }
    uint32_t it = 0;
    for (int w = w0; w < total; w += wstride, ++it) {
      const uint32_t ph = it & 1u;
      int qt, h, v;
      decode(w, qt, h, v);
      const int q0 = qt * QT;
      const int rows = min(QT, Q - q0);
      const int wn = w + wstride;
      float e[32];
      mbar_wait(bar_s, ph);
      tcgen05_fence_after();
      if (active) {
        uint32_t r[32];
        const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(chalf * QT);
        asm volatile(
            "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
            "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
            "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
            : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
              "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
              "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
              "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
            : "r"(taddr)
            : "memory");
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
        for (int c = 0; c < 32; ++c) e[c] = 20.f * __uint_as_float(r[c]);          // a = softmax(20 S)  (gauss:289)
      }
      // the score MMAs are complete (bar_s): the q tiles can take the next item's queries
      if (wn < total) store_q_tiles(sm + L_::QH_OFF, sm + L_::QL_OFF, qnext, tid);
      tcgen05_fence_before();
      mbar_arrive(bar_q);
      // ---- column maxima over the basis rows
      if (active) {
        float t[32];
#pragma unroll
        for (int c = 0; c < 32; ++c) t[c] = e[c];
        wmax[warp * 32 + lane] = warp_transpose_reduce(t, lane, [](float a, float b) { return fmaxf(a, b); });
      }
      cw_sync();
      if (active) {
        float M = -INFINITY;
#pragma unroll
        for (int ww = 0; ww < JWARPS; ++ww) M = fmaxf(M, wmax[ww * 32 + lane]);
#pragma unroll
        for (int c = 0; c < 32; ++c) e[c] = expf(e[c] - __shfl_sync(0xffffffffu, M, c));
        // ---- sum_j e, sum_j e mu_b, sum_j e (mu_b^2 + sigma_b^2): fp64 sums of the fp32 products
        // (the normaliser in fp32: its rounding scales mu and E[t^2] alike and moves var by ~1e-8 at most)
        {
          float tz[32];
#pragma unroll
          for (int c = 0; c < 32; ++c) tz[c] = e[c];
          psum[(0 * 8 + warp) * 32 + lane] =
              (double)warp_transpose_reduce(tz, lane, [](float a, float b) { return a + b; });
        }
        double t[32];
        auto add = [](double a, double b) { return a + b; };
#pragma unroll
        for (int c = 0; c < 32; ++c) t[c] = (double)e[c] * (double)bm;
        psum[(1 * 8 + warp) * 32 + lane] = warp_transpose_reduce(t, lane, add);
#pragma unroll
        for (int c = 0; c < 32; ++c) t[c] = (double)e[c] * (double)c2;
        psum[(2 * 8 + warp) * 32 + lane] = warp_transpose_reduce(t, lane, add);
      }
      cw_sync();
      if (warp == 0) {
        // one thread per query column: mu, var, the canonical-parameter round trip of the reference (gauss:308-310)
        double z = 0.0, am = 0.0, a2 = 0.0;
#pragma unroll
        for (int ww = 0; ww < JWARPS; ++ww) {
          z += psum[(0 * 8 + ww) * 32 + lane];
          am += psum[(1 * 8 + ww) * 32 + lane];
          a2 += psum[(2 * 8 + ww) * 32 + lane];
        }
        const float mu = (float)(am / z);
        const float var = __fsub_rn((float)(a2 / z), __fmul_rn(mu, mu));
        if (lane < rows) {
          const size_t o = (size_t)v * H * Q + (size_t)h * Q + q0 + lane;
          if (p.mu_out) p.mu_out[o] = mu;
          if (p.sd_out) p.sd_out[o] = sqrtf(var);
        }
        const float th0 = __fdiv_rn(mu, var);
        const float th1 = __fdiv_rn(-1.f, __fmul_rn(2.f, var));
        const float var_rt = __fdiv_rn(-0.5f, th1);
        murt[lane] = __fmul_rn(th0, var_rt);
        varrt[lane] = var_rt;
      }
      cw_sync();
      if (active) {
        // r^T element (q = c, j) as hi + lo fp16: k-block j >> 6, row c, 16-byte chunk ((j & 63) >> 3) ^ (c & 7), half j & 7
        uint8_t* rh = sm + L_::RH_OFF + (j >> 6) * 4096 + (lane & 7) * 2;
        uint8_t* rl = sm + L_::RL_OFF + (j >> 6) * 4096 + (lane & 7) * 2;
        const int jchunk = (j & 63) >> 3;
#pragma unroll
        for (int c = 0; c < 32; ++c) {
          // N(mu; mu_b, sigma_b^2 + var) with one reciprocal square root (2 ulp; the reference divides twice)
          const float rs = rsqrtf(__fadd_rn(bs2, varrt[c]));
          const float zz = (murt[c] - bm) * rs;
          const float r = 0.3989422804014327f * __expf(-0.5f * zz * zz) * rs;
          const __half hh = __float2half_rn(r);
          const int off = c * 128 + ((jchunk ^ (c & 7)) << 4);
          *reinterpret_cast<__half*>(rh + off) = hh;
          *reinterpret_cast<__half*>(rl + off) = __float2half_rn(r - __half2float(hh));
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      }
      tcgen05_fence_before();
      mbar_arrive(bar_r);
      if (wn + wstride < total) {                      // queries of item it + 2: consumed after the next bar_s
        int qtn, hn, vn;
        decode(wn + wstride, qtn, hn, vn);
        qnext = load_q(p.q + ((size_t)vn * Q + qtn * QT) * D + hn * DH, min(QT, Q - qtn * QT), D, tid);
      }

      // ---- outputs: D[lane d][q] of the two issuers' accumulators; warp (quarter < 2, chalf) reads 16 columns
      mbar_wait(bar_pv, ph);
      tcgen05_fence_after();
      if (quarter < 2) {
        float dv[16];
        uint32_t r[16], r2[16];
        const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + 64u + (uint32_t)(chalf * 16);
        asm volatile(
            "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
            "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
            : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
              "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
            : "r"(taddr)
            : "memory");
        asm volatile(
            "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
            "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
            : "=r"(r2[0]), "=r"(r2[1]), "=r"(r2[2]), "=r"(r2[3]), "=r"(r2[4]), "=r"(r2[5]), "=r"(r2[6]), "=r"(r2[7]),
              "=r"(r2[8]), "=r"(r2[9]), "=r"(r2[10]), "=r"(r2[11]), "=r"(r2[12]), "=r"(r2[13]), "=r"(r2[14]),
              "=r"(r2[15])
            : "r"(taddr + 32u)
            : "memory");
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
        for (int i = 0; i < 16; ++i) dv[i] = __uint_as_float(r[i]) + __uint_as_float(r2[i]);
        const int dd = quarter * 32 + lane;
        float* dst = p.ctx + ((size_t)v * Q + q0 + chalf * 16) * D + h * DH + dd;
#pragma unroll
        for (int i = 0; i < 16; ++i)
          if (chalf * 16 + i < rows) dst[(size_t)i * D] = dv[i];
      }
      // (no barrier before the next item: wmax / psum / murt are rewritten only behind the next item's cw_syncs, which
      // no thread passes before all of them have finished reading this item's values)
    }
  }
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 8) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)TMEM_COLS)
                 : "memory");
  }
}

template <int NB>
static int launch(const CUtensorMap& mKh, const CUtensorMap& mKl, const CUtensorMap& mVh, const CUtensorMap& mVl,
                  const Params& p, int Bv, cudaStream_t stream) {
  static PerDevice pd = {};
  int num_sms = 0;
  if (int rc = kernel_setup(cont_attn_g16_kernel<NB>, (size_t)Lay<NB>::BYTES, pd, &num_sms)) return rc;
  const int q_tiles = (p.Q + QT - 1) / QT;
  const long long total = (long long)q_tiles * p.H * Bv;
  LTM_REQUIRE(total < (1ll << 31), "cont_attn_gauss_tc16: too many work items");
  const unsigned grid = (unsigned)(total < num_sms ? total : num_sms);       // persistent: one CTA per SM
  cont_attn_g16_kernel<NB><<<grid, THREADS, Lay<NB>::BYTES, stream>>>(mKh, mKl, mVh, mVl, p, q_tiles, (int)total);
  LTM_CHECK_LAUNCH("cont_attn_gauss_tc16");
  return 0;
}

}  // namespace g16
}  // namespace ltm

extern "C" int ltm_cont_attn_gauss_tc16(const float* q, const void* KV_hi, const void* KV_lo, int64_t ldkv,
                                        const float* basis_mu, const float* basis_sigma, float* ctx, float* mu_out,
                                        float* sd_out, int Bv, int Q, int N, int H, int d, void* stream) {
  using namespace ltm;
  LTM_REQUIRE(q && KV_hi && KV_lo && basis_mu && basis_sigma && ctx, "cont_attn_gauss_tc16: null pointer");
  LTM_REQUIRE(ltm_attn_tc_supported(N, d), "cont_attn_gauss_tc16: unsupported num_basis=%d / head_size=%d", N, d);
  LTM_REQUIRE(Bv > 0 && Bv <= 65535 && Q > 0 && H > 0 && H <= 65535 && ldkv % 8 == 0 && ldkv >= 2 * (int64_t)H * d,
              "cont_attn_gauss_tc16: bad shape");
  LTM_REQUIRE(aligned16(q) && aligned16(ctx), "cont_attn_gauss_tc16: 16-byte alignment");
  const unsigned long long rows = (unsigned long long)Bv * N, hd = (unsigned long long)H * d;
  const uint16_t* kh = reinterpret_cast<const uint16_t*>(KV_hi);
  const uint16_t* kl = reinterpret_cast<const uint16_t*>(KV_lo);
  CUtensorMap mKh, mKl, mVh, mVl;
  if (tma_encode_2d_f16(&mKh, kh, hd, rows, (unsigned long long)ldkv, (unsigned)N, "attn_g16 K hi")) return -1;
  if (tma_encode_2d_f16(&mKl, kl, hd, rows, (unsigned long long)ldkv, (unsigned)N, "attn_g16 K lo")) return -1;
  if (tma_encode_2d_f16(&mVh, kh + hd, hd, rows, (unsigned long long)ldkv, (unsigned)N, "attn_g16 V hi")) return -1;
  if (tma_encode_2d_f16(&mVl, kl + hd, hd, rows, (unsigned long long)ldkv, (unsigned)N, "attn_g16 V lo")) return -1;
  g16::Params p{};
  p.q = q; p.bmu = basis_mu; p.bsig = basis_sigma; p.ctx = ctx; p.mu_out = mu_out; p.sd_out = sd_out;
  p.Q = Q; p.H = H;
  if (N == 256) return g16::launch<256>(mKh, mKl, mVh, mVl, p, Bv, (cudaStream_t)stream);
  if (N == 128) return g16::launch<128>(mKh, mKl, mVh, mVl, p, Bv, (cudaStream_t)stream);
  return g16::launch<64>(mKh, mKl, mVh, mVl, p, Bv, (cudaStream_t)stream);
}
