// Continuous attention over rectangular bases (R10/R11 + R6) on the tcgen05 tensor cores.
// long_term_attention_gibbs.py:224-286 (expected value by quadrature), :196-203 (sticky histogram of the next call).
//
// Same mathematics as attn.cu / attn_fast.cu (closed form of the 1000-point quadrature,
// r_j = W_j e^{S_j} / (sum_i W_i e^{S_i} + W_out)), but both contractions run as tf32 UMMAs with the basis index j
// on the TMEM lanes, one CTA per (query tile of 32, head, video):
//
//   S^T[j, q] = K_h[j, :] . q_h[q, :]          A = K_h  (TMA, K-major, SWIZZLE_128B, [NB j][64 d]),
//                                              B = q_h/sqrt(d) rounded to tf32, written by the CTA (K-major)
//   thread j:  e[q] = W_j exp(S[j,q] - m_q),   m_q = max(0, max_j S[j,q])  (redux.sync + one smem exchange)
//   D[m, q]   = sum_j A2[m, j] e[j, q]         A2 = [V_h^T ; X^T ; *]  (TMA, MN-major, SWIZZLE_128B_ATOM_32B):
//                 rows  0..63  V_h[:, d]                 -> un-normalised context
//                 row   64     1                         -> quadrature normaliser  sum_j e[j,q]
//                 rows  65,66  c_j / W_j  (hi, lo)       -> trapezoid integral of the sticky-edge density
//               B = e^T rounded to tf32, written by the CTA in the K-major SWIZZLE_128B layout
//   ctx[q, d]  = D[d, q] / (D[64, q] + W_out e^{-m_q})
//   histogram: p_i = dt_{i+1}/2 (G[jb_{i+1}] + G[jb_{i+2}]),  G[j] = sum_q exp(S[j,q] - m_q) / Z_q  -- the per-row
//              trapezoid of rect_hist.cuh regrouped by basis (every edge value is the weight of one basis or of
//              "no basis"), so no cross-thread reduction is left: the column sums come out of the tensor core.
//
// The FMA kernels spend 2 x 524 k FMAs per CTA on 85 registers x 768 threads per SM; here the SM's register file
// and issue slots stay almost free (288 threads), which is what lets the frame pooling of the next chunk run
// beside it (BatchedRectLTM.prefetch).  K and V must already be tf32-rounded (ltm_gemm round_tf32) so that the
// tensor core's own fp32 -> tf32 truncation does not bias the scores.
//
// K|V stored as fp16 (KvF16, the default) run the same kernel with another operand format: K|V come in as IEEE fp16
// -- the same 11-bit significand as the tf32 grid, at half the bytes -- the queries and the attention weights are
// written as fp16 by the CTA, and both contractions run as kind::f16 UMMAs (K = 16 per instruction) with fp32
// accumulation in TMEM:
//
//   S^T[j, q] = K_h[j, :] . q_h[q, :]     A = K_h  (TMA, K-major SWIZZLE_128B: one row of 64 halves = 128 B per basis)
//                                          B = q_h / sqrt(d) as fp16, written by the CTA ([32 q][64 d], K-major)
//   D[m, q]   = sum_j A2[m, j] e[j, q]    A2 = [V_h^T ; X^T] (TMA, MN-major SWIZZLE_128B: atoms of 8 j-rows x 64 halves;
//                                          the 64 value columns and the 64-column table X are the two MN atoms, so
//                                          M = 128 exactly), B = e^T as fp16 ([NB/64 k-blocks][32 q][64 j], K-major)
//
// The fp16 weights are scaled by 256 (e' = 256 W_j exp(S - m), W_j ~ 1/256: the largest weight is ~1) so that weights
// down to e^{-9.7} of the largest stay fp16-normal; the factor cancels in every ratio that leaves the kernel.
// Shared memory per CTA at num_basis 256: K 32 KB + V 32 KB + X 32 KB + e^T 16 KB + q 4 KB (fp32 K|V: 200 KB).
#include <cuda_fp16.h>

#include "rect_hist.cuh"
#include "tcgen05.cuh"

namespace ltm {
namespace tc {

constexpr int DH = 64;
constexpr int QT = 32;
constexpr int THREADS = 320;             // 8 compute warps (TMEM lane quarter = warp % 4) + 2 issuing warps
// register cap: 320 threads x 96 leave room for three frame-pooling CTAs of the next chunk beside this kernel
constexpr int TC_MAX_REGS = 96;
constexpr int TMEM_COLS = 128;           // S^T: NB/128 x 32 columns at 0; D: 2 x 32 columns at 64 (one per issuer)

struct Params {
  const float* q;        // [Bv,Q,D]
  const float* W;        // [NB] quadrature weight per basis
  const float* tb;       // [129] sticky edges
  const int32_t* jb;     // [129] basis at each edge (-1: none)
  float W_out, c_none;
  float* ctx;            // [Bv,Q,D]
  float* scores_out;     // optional [Bv,H,Q,NB]
  float* hist_part;      // optional [Bv, H*q_tiles, 127]
  int Q, H;
  // num_basis = halves * NB: with halves == 2 (num_basis 512) every (query tile, head, video) is two work items, one
  // per half of the basis range; each writes its un-normalised accumulator rows, the normaliser sums and its shift
  // m_q to `part` ([item][68][32]: rows 0..63 D[d][q], 64 sum_j e, 65 / 66 the histogram integral hi / lo, 67 m_q)
  // and attn_tc_combine_kernel merges the two halves (exp(m_half - m) rescaling, as in a two-block online softmax).
  int halves, NT;
  float* part;
};
constexpr int PART_ROWS = 68;

// Storage formats of K|V.  ROW: elements in one 128-byte swizzle row, so that every UMMA consumes 32 bytes of K
// (ROW / 4 elements); V_SBO / V_LAYOUT: UMMA descriptor of the MN-major A2 operand.
struct KvTf32 {                          // fp32 on the tf32 grid: kind::tf32, A2 in SWIZZLE_128B_BASE32B
  static constexpr bool HALF = false;
  static constexpr int ROW = 32;
  static constexpr uint32_t IDESC_AB = (2u << 7) | (2u << 10);
  static constexpr uint32_t V_SBO = 512, V_LAYOUT = 1;
  static constexpr float WSCALE = 1.f;
  static constexpr const char* NAME = "cont_attn_rect_tc";
};
struct KvF16 {                           // IEEE fp16: kind::f16, A2 in 16-bit SWIZZLE_128B (atoms of [8 j][64 mn])
  static constexpr bool HALF = true;
  static constexpr int ROW = 64;
  static constexpr uint32_t IDESC_AB = 0u;
  static constexpr uint32_t V_SBO = 1024, V_LAYOUT = 2;
  static constexpr float WSCALE = 256.f; // weights are formed as 256 W_j exp(S - m): fp16-normal down to e^{-9.7}
  static constexpr const char* NAME = "cont_attn_rect_tc16";
};

template <int NB, class KV>
struct Lay {
  static constexpr int SLAB = NB * 128;              // NB rows x 128 B: 32 floats or 64 halves
  static constexpr int KSLABS = DH / KV::ROW;        // slabs of one K|V row: 2 (d 0..31 | d 32..63) or 1
  static constexpr int K_OFF = 0;                    // KSLABS slabs: K_h                 (K-major rows = j)
  static constexpr int V_OFF = KSLABS * SLAB;        // KSLABS + 1 slabs: V_h | X         (MN-major rows = j)
  static constexpr int R_OFF = V_OFF + (KSLABS + 1) * SLAB;   // e^T: [NB/ROW k-blocks][32 q][ROW j]; fp32: also
                                                              // "slab 3" of A2
  static constexpr int R_BYTES = ((NB + KV::ROW - 1) / KV::ROW) * 4096;   // (fp16, NB = 64: one block)
  static constexpr int Q_OFF = R_OFF + R_BYTES;      // q tile: [KSLABS k-blocks][32 q][ROW d]
  static constexpr int MISC_OFF = Q_OFF + KSLABS * 4096;
  static constexpr int MISC_FLOATS = 8 * 32 + 4 * 32 + 96 + NB + 32;
  static constexpr int BYTES = MISC_OFF + MISC_FLOATS * 4 + 64 + 1024;   // + 6 barriers, TMEM slot, alignment slack
};

template <class KV>
__device__ __forceinline__ void mma(uint32_t tmem_d, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi,
                                    uint32_t idesc, uint32_t accumulate) {
  if constexpr (KV::HALF)
    tcgen05_mma_f16(tmem_d, a_lo, a_hi, b_lo, b_hi, idesc, accumulate);
  else
    tcgen05_mma_tf32(tmem_d, a_lo, a_hi, b_lo, b_hi, idesc, accumulate);
}

__device__ __forceinline__ void cw_sync() { asm volatile("bar.sync 1, 256;" ::: "memory"); }   // the 8 compute warps

// q tile of one work item, scaled by 1/sqrt(d) (gibbs:226; a power of two, exact) and rounded to the operand format,
// in the K-major SWIZZLE_128B layout.  tf32: element (q, d) at [d >> 5][q][((d & 31) >> 2) ^ (q & 7)][d & 3]; fp16:
// row q = 64 halves = 128 B, 16-byte chunk (d >> 3) at position (d >> 3) ^ (q & 7).  256 threads, 8 consecutive d
// each; the global loads are issued one item ahead (load_q) so that their latency is off the item's critical path.
struct QRegs { float4 a, b; };
__device__ __forceinline__ QRegs load_q(const float* qbase, int rows, int D, int tid) {
  const int qq = tid >> 3, dch = tid & 7;                          // 8 consecutive d per thread
  QRegs r;
  r.a = make_float4(0.f, 0.f, 0.f, 0.f);
  r.b = r.a;
  if (qq < rows) {
    // volatile asm: the loads stay where they are written (one item ahead of their use) instead of being sunk
    // next to the first use by the scheduler
    const float4* src = reinterpret_cast<const float4*>(qbase + (size_t)qq * D + dch * 8);
    asm volatile("ld.global.nc.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(r.a.x), "=f"(r.a.y), "=f"(r.a.z), "=f"(r.a.w) : "l"(src));
    asm volatile("ld.global.nc.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(r.b.x), "=f"(r.b.y), "=f"(r.b.z), "=f"(r.b.w) : "l"(src + 1));
  }
  return r;
}
__device__ __forceinline__ uint32_t pack_h2(float lo, float hi) {
  const __half2 h = __floats2half2_rn(lo, hi);
  return *reinterpret_cast<const uint32_t*>(&h);
}
template <class KV>
__device__ __forceinline__ void store_q_tile(uint8_t* dstq, const QRegs& r, int tid) {
  const int qq = tid >> 3, dch = tid & 7;
  const float sc = 0.125f;
  if constexpr (KV::HALF) {
    const uint4 v = make_uint4(pack_h2(r.a.x * sc, r.a.y * sc), pack_h2(r.a.z * sc, r.a.w * sc),
                               pack_h2(r.b.x * sc, r.b.y * sc), pack_h2(r.b.z * sc, r.b.w * sc));
    *reinterpret_cast<uint4*>(dstq + qq * 128 + ((dch ^ (qq & 7)) << 4)) = v;
  } else {
    const float4 a = make_float4(tf32_rna(r.a.x * sc), tf32_rna(r.a.y * sc), tf32_rna(r.a.z * sc), tf32_rna(r.a.w * sc));
    const float4 b = make_float4(tf32_rna(r.b.x * sc), tf32_rna(r.b.y * sc), tf32_rna(r.b.z * sc), tf32_rna(r.b.w * sc));
    uint8_t* row = dstq + (dch >> 2) * 4096 + qq * 128;
    const int c0 = (dch & 3) * 2;
    *reinterpret_cast<float4*>(row + (((c0) ^ (qq & 7)) << 4)) = a;
    *reinterpret_cast<float4*>(row + (((c0 + 1) ^ (qq & 7)) << 4)) = b;
  }
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

// Persistent: CTA b walks the work items w = b, b + grid, ... (w -> query tile, head, video; head fastest).
// Per item, warp 8 (one lane) issues  S MMAs -> [K buffer free] TMA K(next) -> PV MMAs -> [V buffer free] TMA V(next)
// and the 8 compute warps run  read S -> write q(next) -> weights -> write e^T -> read D -> outputs,  so the next
// item's keys land during this item's weight phase and its values during the output phase + the next score MMAs.
//   bar_k / bar_v   TMA bytes of this item's K / V (+ X once)            bar_s / bar_pv   tcgen05.commit
//   bar_q           256 arrivals: q tile of the next item is in place (and S has been read out of TMEM)
//   bar_r           256 arrivals: e^T is in place (and D of the previous item has been read out of TMEM)
template <int NB, class KV>
__global__ void __maxnreg__(TC_MAX_REGS)
cont_attn_tc_kernel(const __grid_constant__ CUtensorMap mapK, const __grid_constant__ CUtensorMap mapV,
                    const __grid_constant__ CUtensorMap mapX, const Params p, const int q_tiles, const int total) {
  static_assert(NB == 64 || NB == 128 || NB == 256, "the tensor-core path covers num_basis 64 / 128 / 256");
  using L_ = Lay<NB, KV>;
  constexpr int KSLABS = L_::KSLABS;
  constexpr int MMA_K = KV::ROW / 4;         // elements of K per UMMA: 32 bytes, a quarter of a swizzle row
  constexpr int HALVES = (NB + 127) / 128;   // score MMAs (M = 128 each); NB = 64: the upper 64 rows read past the
                                             // K tile (finite or not, they only reach accumulator rows nobody reads)
  constexpr int JWARPS = NB / 32;            // compute warps that own a basis (the others only help with the outputs)
  extern __shared__ uint8_t smem_raw[];
  const uint32_t sbase = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* sm = smem_raw + (sbase - smem_u32(smem_raw));
  float* misc = reinterpret_cast<float*>(sm + L_::MISC_OFF);
  float* wmax = misc;                       // [8][32]
  float* mcol = wmax + 8 * 32;              // [32]
  float* zq = mcol + 32;                    // [32] reciprocal of the quadrature normaliser
  float* rzh = zq + 32;                     // [32]
  float* ems = rzh + 32;                    // [32] e^{-m_q} / Z_q (histogram)
  float* nrm = ems + 32;                    // [2][3][16] scratch of the normaliser rows
  float* Gs = nrm + 96;                     // [NB + 1]
  const uint32_t bars = sbase + L_::MISC_OFF + L_::MISC_FLOATS * 4;
  const uint32_t bar_k = bars, bar_v = bars + 8, bar_s = bars + 16, bar_pv = bars + 24, bar_q = bars + 32,
                 bar_r = bars + 40;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(sm + L_::MISC_OFF + L_::MISC_FLOATS * 4 + 48);

  const int Q = p.Q, H = p.H, D = H * DH;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t sK = sbase + L_::K_OFF, sV = sbase + L_::V_OFF, sR = sbase + L_::R_OFF, sQ = sbase + L_::Q_OFF;
  // videos are walked last-to-first: the projection kernel that ran just before wrote K|V first-to-last, so the
  // most recently written rows are the ones still resident in L2
  const int halves = p.halves, NT = p.NT;
  const int nvid = total / (H * q_tiles * halves);
  // (qt, h, v) of a work item; the basis half is w % halves and enters through `jrow` = first K|V row of the item
  auto decode = [&](int w, int& qt, int& h, int& v) {
    const int w2 = w / halves;
    h = w2 % H;
    qt = (w2 / H) % q_tiles;
    v = nvid - 1 - w2 / (H * q_tiles);
  };
  auto jrow = [&](int w, int v) { return v * NT + (w % halves) * NB; };
  const int w0 = blockIdx.x, wstride = gridDim.x;

  if (warp == 8) {
    if (lane == 0) {
      asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&mapK)) : "memory");
      asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&mapV)) : "memory");
      asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&mapX)) : "memory");
      mbar_init(bar_k, 1);
      mbar_init(bar_v, 1);
      mbar_init(bar_s, 1);
      mbar_init(bar_pv, 2);                            // one commit per issuing warp
      mbar_init(bar_q, 256);
      mbar_init(bar_r, 256);
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
      int qt, h, v;
      decode(w0, qt, h, v);
      mbar_arrive_expect_tx(bar_k, KSLABS * L_::SLAB);
      tma_load_2d(&mapK, sK, bar_k, h * DH, jrow(w0, v));
      if constexpr (KSLABS == 2) tma_load_2d(&mapK, sK + L_::SLAB, bar_k, h * DH + 32, jrow(w0, v));
      mbar_arrive_expect_tx(bar_v, (KSLABS + 1) * L_::SLAB);
      tma_load_2d(&mapV, sV, bar_v, h * DH, jrow(w0, v));
      if constexpr (KSLABS == 2) tma_load_2d(&mapV, sV + L_::SLAB, bar_v, h * DH + 32, jrow(w0, v));
      tma_load_2d(&mapX, sV + KSLABS * L_::SLAB, bar_v, 0, (w0 % halves) * NB);
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

  // instruction descriptors: D=f32 [4,6)=1, A [7,10) and B [10,13) = KV::IDESC_AB (tf32 2, f16 0), a_major bit 15
  // (1 = MN-major), N>>3 [17,23), M>>4 [24,29)
  constexpr uint32_t IDESC_S = (1u << 4) | KV::IDESC_AB | ((uint32_t)(QT >> 3) << 17) | ((128u >> 4) << 24);
  constexpr uint32_t IDESC_PV = IDESC_S | (1u << 15);

  if (warp == 8) {
    // ------------------------------------------------------------------ TMA + MMA issue (one lane)
    if (lane == 0) {
      // descriptor words: only the start-address field of the low word changes between MMAs (compile-time offsets)
      // K-major SWIZZLE_128B: 8-row groups 1024 B apart; MN-major A2: the MN atoms one slab apart (LBO), the 8-row j
      // groups KV::V_SBO apart; an MMA of K = MMA_K consumes MMA_K rows of j
      const uint64_t dK = umma_desc(sK, 16, 1024, 2u), dQ = umma_desc(sQ, 16, 1024, 2u);
      const uint64_t dV = umma_desc(sV, L_::SLAB, KV::V_SBO, KV::V_LAYOUT), dR = umma_desc(sR, 16, 1024, 2u);
      const uint32_t dk_lo = (uint32_t)dK, dk_hi = (uint32_t)(dK >> 32), dq_lo = (uint32_t)dQ;
      const uint32_t dv_lo = (uint32_t)dV, dv_hi = (uint32_t)(dV >> 32), dr_lo = (uint32_t)dR;
      auto issue_scores = [&](uint32_t ph) {            // S^T of the item whose K tile / q tile carry parity ph
        mbar_wait(bar_q, ph);                          // q tile written, S read out of TMEM
        mbar_wait(bar_k, ph);
        tcgen05_fence_after();
#pragma unroll
        for (int hf = 0; hf < HALVES; ++hf) {
#pragma unroll
          for (int ks = 0; ks < DH / MMA_K; ++ks)      // (ks >> 2: second slab of K / k-block of q, fp32 only)
            mma<KV>(tmem_base + hf * QT,
                    dk_lo + (uint32_t)(((ks >> 2) * L_::SLAB + hf * (128 * 128) + (ks & 3) * 32) >> 4), dk_hi,
                    dq_lo + (uint32_t)(((ks >> 2) * 4096 + (ks & 3) * 32) >> 4), dk_hi, IDESC_S, ks != 0 ? 1u : 0u);
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
        mbar_wait(bar_s, ph);                          // the K buffer has been read
        if (wn < total) {
          mbar_arrive_expect_tx(bar_k, KSLABS * L_::SLAB);
          tma_load_2d(&mapK, sK, bar_k, hn * DH, jrow(wn, vn));
          if constexpr (KSLABS == 2) tma_load_2d(&mapK, sK + L_::SLAB, bar_k, hn * DH + 32, jrow(wn, vn));
        }
        mbar_wait(bar_r, ph);                          // e^T written, D free
        mbar_wait(bar_v, ph);
        tcgen05_fence_after();
        // this warp contracts the first half of the basis range into D0, warp 9 the second half into D1: the issue
        // of 32 small MMAs by one thread (~33 ns each) was 1.05 us of the item's 4.7 us
#pragma unroll
        for (int ks = 0; ks < NB / (2 * MMA_K); ++ks)
          mma<KV>(tmem_base + 64, dv_lo + (uint32_t)((ks * MMA_K * 128) >> 4), dv_hi,
                  dr_lo + (uint32_t)(((ks >> 2) * 4096 + (ks & 3) * 32) >> 4), dk_hi, IDESC_PV, ks != 0 ? 1u : 0u);
        tcgen05_commit(bar_pv);
        // the next item's scores go out right behind: its keys landed during this item's weight phase, so S is
        // ready by the time the compute warps have written this item's outputs
        if (wn < total) issue_scores(ph ^ 1u);
        mbar_wait(bar_pv, ph);                         // the V buffer (and e^T) have been read
        if (wn < total) {
          // (the per-basis operand rows X change with the basis half: re-fetched with V when there are two)
          mbar_arrive_expect_tx(bar_v, (halves > 1 ? KSLABS + 1 : KSLABS) * L_::SLAB);
          tma_load_2d(&mapV, sV, bar_v, hn * DH, jrow(wn, vn));
          if constexpr (KSLABS == 2) tma_load_2d(&mapV, sV + L_::SLAB, bar_v, hn * DH + 32, jrow(wn, vn));
          if (halves > 1) tma_load_2d(&mapX, sV + KSLABS * L_::SLAB, bar_v, 0, (wn % halves) * NB);
        }
      }
    }
    __syncwarp();
  } else if (warp == 9) {
    // ------------------------------------------------------------------ second MMA issuer (one lane)
    if (lane == 0) {
      const uint64_t dV = umma_desc(sV, L_::SLAB, KV::V_SBO, KV::V_LAYOUT), dR = umma_desc(sR, 16, 1024, 2u);
      const uint32_t dv_lo = (uint32_t)dV, dv_hi = (uint32_t)(dV >> 32), dr_lo = (uint32_t)dR, dr_hi = (uint32_t)(dR >> 32);
      uint32_t it = 0;
      for (int w = w0; w < total; w += wstride, ++it) {
        const uint32_t ph = it & 1u;
        mbar_wait(bar_r, ph);
        mbar_wait(bar_v, ph);
        tcgen05_fence_after();
#pragma unroll
        for (int ks = NB / (2 * MMA_K); ks < NB / MMA_K; ++ks)
          mma<KV>(tmem_base + 96, dv_lo + (uint32_t)((ks * MMA_K * 128) >> 4), dv_hi,
                  dr_lo + (uint32_t)(((ks >> 2) * 4096 + (ks & 3) * 32) >> 4), dr_hi, IDESC_PV,
                  ks != NB / (2 * MMA_K) ? 1u : 0u);
        tcgen05_commit(bar_pv);
      }
    }
    __syncwarp();
  } else {
    // ------------------------------------------------------------------ compute warps
    const bool active = warp < JWARPS;
    const int j = (warp >> 2) * 128 + (warp & 3) * 32 + lane;      // this thread's basis in the weight phase
    const int quarter = warp & 3, chalf = warp >> 2;
    float Wj = active ? KV::WSCALE * __ldg(p.W + (w0 % halves) * NB + j) : 0.f;
    float rWj = active ? 1.0f / Wj : 0.f;
    // histogram bin of this thread (tid < 127): p_i = dt_{i+1}/2 (G[jb_{i+1}] + G[jb_{i+2}])
    int hja = NB, hjb = NB;
    float hdt = 0.f;
    if (tid < EDGES - 2 && p.hist_part != nullptr) {
      const int a = __ldg(p.jb + tid + 1), b = __ldg(p.jb + tid + 2);
      hja = a < 0 ? NB : a;
      hjb = b < 0 ? NB : b;
      hdt = 0.5f * (__ldg(p.tb + tid + 2) - __ldg(p.tb + tid + 1));
    }
    {
      int qt, h, v;
      decode(w0, qt, h, v);
      const QRegs qr = load_q(p.q + ((size_t)v * Q + qt * QT) * D + h * DH, min(QT, Q - qt * QT), D, tid);
      store_q_tile<KV>(sm + L_::Q_OFF, qr, tid);
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
      float e[32];
      const int wn = w + wstride;
      const int jhalf = (w % halves) * NB;               // first basis of this item's half
      if (halves > 1 && active) {
        Wj = KV::WSCALE * __ldg(p.W + jhalf + j);
        rWj = 1.0f / Wj;
      }
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
        for (int c = 0; c < 32; ++c) e[c] = __uint_as_float(r[c]);
      }
      // the score MMAs are complete (bar_s): the q tile can take the next item's queries
      if (wn < total) store_q_tile<KV>(sm + L_::Q_OFF, qnext, tid);
      tcgen05_fence_before();
      mbar_arrive(bar_q);
      if (active) {
        uint32_t mine = 0u;
#pragma unroll
        for (int c = 0; c < 32; ++c) {
          // non-negative floats order like their bit patterns: one redux.sync per column
          const uint32_t mx = __reduce_max_sync(0xffffffffu, __float_as_uint(fmaxf(e[c], 0.f)));
          if (lane == c) mine = mx;
        }
        wmax[warp * 32 + lane] = __uint_as_float(mine);
        if (p.scores_out) {
          float* dst = p.scores_out + (((size_t)v * H + h) * Q + q0) * NT + jhalf + j;
#pragma unroll
          for (int c = 0; c < 32; ++c)
            if (c < rows) dst[(size_t)c * NT] = e[c];
        }
      }
      cw_sync();                                                                           // column maxima
      if (active) {
        float M = 0.f;                                 // per-row shift m = max(0, max_j S_j): it cancels exactly
#pragma unroll
        for (int ww = 0; ww < JWARPS; ++ww) M = fmaxf(M, wmax[ww * 32 + lane]);
        if (warp == 0) mcol[lane] = M;
        if constexpr (KV::HALF) {
          // e^T element (q = c, j) as fp16: k-block j >> 6, row c, 16-byte chunk ((j & 63) >> 3) ^ (c & 7), half j & 7
          uint8_t* rblk = sm + L_::R_OFF + (j >> 6) * 4096 + (lane & 7) * 2;
          const int jchunk = (j & 63) >> 3;
#pragma unroll
          for (int c = 0; c < 32; ++c) {
            const float m = __shfl_sync(0xffffffffu, M, c);
            e[c] = Wj * __expf(e[c] - m);
            *reinterpret_cast<__half*>(rblk + c * 128 + ((jchunk ^ (c & 7)) << 4)) = __float2half_rn(e[c]);
          }
        } else {
          uint8_t* rblk = sm + L_::R_OFF + (j >> 5) * 4096 + (lane & 3) * 4;
#pragma unroll
          for (int c = 0; c < 32; ++c) {
            const float m = __shfl_sync(0xffffffffu, M, c);
            e[c] = Wj * __expf(e[c] - m);
            // e^T element (q = c, j): row c of k-block j >> 5, chunk ((j & 31) >> 2) ^ (c & 7)
            *reinterpret_cast<float*>(rblk + c * 128 + ((((lane >> 2) ^ (c & 7))) << 4)) = tf32_rna(e[c]);
          }
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

      // ---- outputs: D[lane m][q]; warp (quarter, chalf) reads 16 columns
      mbar_wait(bar_pv, ph);
      tcgen05_fence_after();
      float dv[16];
      {
        uint32_t r[16];
        const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + 64u + (uint32_t)(chalf * 16);
        asm volatile(
            "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
            "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
            : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
              "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
            : "r"(taddr)
            : "memory");
        uint32_t r2[16];
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
      }
      if (p.part != nullptr) {
        // one half of a two-half item: hand the raw accumulator rows, the normaliser sums and the shift to the combine
        // kernel (TMEM lane = row m: quarters 0, 1 hold D[d][q], lanes 0..2 of quarter 2 the three sums)
        float* pw = p.part + (size_t)w * (PART_ROWS * QT);
        const int prow = quarter * 32 + lane;
        if (quarter < 2 || (quarter == 2 && lane < 3)) {
          float4* dst = reinterpret_cast<float4*>(pw + prow * QT + chalf * 16);
#pragma unroll
          for (int i = 0; i < 4; ++i) dst[i] = make_float4(dv[4 * i], dv[4 * i + 1], dv[4 * i + 2], dv[4 * i + 3]);
        }
        if (quarter == 3 && lane < 16) pw[67 * QT + chalf * 16 + lane] = mcol[chalf * 16 + lane];
        continue;    // (mcol is rewritten behind the next item's first cw_sync, which every thread must reach first)
      }
      if (quarter == 2) {
        // lanes 0,1,2 hold rows 64 (sum_j e), 65, 66 (sum_j c_j/W_j e, hi + lo) of this warp's 16 columns: through
        // a small scratch so that 16 lanes finish one column each
        float* sc = nrm + chalf * 48;
        if (lane < 3) {
#pragma unroll
          for (int i = 0; i < 16; ++i) sc[lane * 16 + i] = dv[i];
        }
        __syncwarp();
        if (lane < 16) {
          const int c = chalf * 16 + lane;
          const float em = expf(-mcol[c]);
          zq[c] = 1.0f / (sc[lane] + KV::WSCALE * p.W_out * em);
          const float rz = (c < rows) ? 1.0f / (sc[16 + lane] + sc[32 + lane] + KV::WSCALE * p.c_none * em) : 0.f;
          rzh[c] = rz;
          ems[c] = em * rz;
        }
      }
      cw_sync();                                                                           // normalisers
      if (quarter < 2) {
        const int dd = quarter * 32 + lane;
        float* dst = p.ctx + ((size_t)v * Q + q0 + chalf * 16) * D + h * DH + dd;
#pragma unroll
        for (int i = 0; i < 16; ++i)
          if (chalf * 16 + i < rows) dst[(size_t)i * D] = dv[i] * zq[chalf * 16 + i];
      }
      if (p.hist_part != nullptr) {
        if (active) {
          // G[j] = sum_q exp(S[j,q] - m_q) / Z_q = (1 / W_j) sum_q e[q] / Z_q
          float g = 0.f;
#pragma unroll
          for (int c = 0; c < 32; ++c) g = fmaf(e[c], rzh[c], g);
          Gs[j] = g * rWj;
        }
        if (warp == 3) {                               // edges outside every basis (score 0): sum_q e^{-m_q} / Z_q
          const float g = warp_sum(ems[lane]);
          if (lane == 0) Gs[NB] = g;
        }
        cw_sync();                                                                         // G complete
        if (tid < EDGES - 2)
          p.hist_part[((size_t)v * (H * q_tiles) + h * q_tiles + qt) * (EDGES - 2) + tid] =
              hdt * (Gs[hja] + Gs[hjb]);
        // no barrier before the next item: everything above is rewritten only behind the next item's first
        // cw_sync, which no thread passes before all of them have finished this item
      }
    }
  }
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 8) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)TMEM_COLS)
                 : "memory");
  }
}

// Merge of the two basis halves of num_basis = 512: ctx = (D_0 s_0 + D_1 s_1) / (Z_0 s_0 + Z_1 s_1 + W_out e^{-m}),
// m = max(m_0, m_1), s_i = e^{m_i - m}.  One CTA per (query tile, head, video); thread -> (q, d) with d fastest.
// W_out is the quadrature weight on the scale of the stored sums (KV::WSCALE * W_out).
__global__ void __launch_bounds__(256)
attn_tc_combine_kernel(const float* __restrict__ part, float* __restrict__ ctx, float W_out, int Q, int H,
                       int q_tiles, int nvid) {
  const int w2 = blockIdx.x;
  const int h = w2 % H, qt = (w2 / H) % q_tiles, v = nvid - 1 - w2 / (H * q_tiles);
  const float* p0 = part + (size_t)(2 * w2) * (PART_ROWS * QT);
  const float* p1 = p0 + PART_ROWS * QT;
  __shared__ float s0[QT], s1[QT], rz[QT];
  if (threadIdx.x < QT) {
    const int q = threadIdx.x;
    const float m0 = p0[67 * QT + q], m1 = p1[67 * QT + q];
    const float m = fmaxf(m0, m1);
    const float a = expf(m0 - m), b = expf(m1 - m);
    s0[q] = a;
    s1[q] = b;
    rz[q] = 1.0f / (p0[64 * QT + q] * a + p1[64 * QT + q] * b + W_out * expf(-m));
  }
  __syncthreads();
  const int q0 = qt * QT, rows = min(QT, Q - q0), D = H * DH;
  for (int i = threadIdx.x; i < QT * DH; i += 256) {
    const int d = i & (DH - 1), q = i >> 6;
    if (q < rows)
      ctx[((size_t)v * Q + q0 + q) * D + h * DH + d] = (p0[d * QT + q] * s0[q] + p1[d * QT + q] * s1[q]) * rz[q];
  }
}

template <int NB, class KV>
static int launch(const CUtensorMap& mK, const CUtensorMap& mV, const CUtensorMap& mX, const Params& p, int Bv,
                  cudaStream_t stream) {
  using L_ = Lay<NB, KV>;
  static PerDevice pd = {};
  int num_sms = 0;
  if (int rc = kernel_setup(cont_attn_tc_kernel<NB, KV>, (size_t)L_::BYTES, pd, &num_sms)) return rc;
  const int q_tiles = (p.Q + QT - 1) / QT;
  const long long total = (long long)q_tiles * p.H * Bv * p.halves;
  LTM_REQUIRE(total < (1ll << 31), "cont_attn_rect_tc: too many work items");
  // persistent CTAs: one per SM for num_basis 256 (209 KB of shared memory), two for 64 / 128 (60 / 106 KB; 2 x 320
  // threads x 96 registers and 2 x 128 TMEM columns fit): an item costs ~3 us of mostly latency whatever its size, so
  // the small shapes (cfg1, cfg3: 12 k / 2.3 k items of 64 bases) gain from a second CTA filling the bubbles
  constexpr int PER_SM = (2 * L_::BYTES <= 227 * 1024) ? 2 : 1;
  const long long slots = (long long)num_sms * PER_SM;
  const unsigned grid = (unsigned)(total < slots ? total : slots);
  cont_attn_tc_kernel<NB, KV><<<grid, THREADS, L_::BYTES, stream>>>(mK, mV, mX, p, q_tiles, (int)total);
  LTM_CHECK_LAUNCH("cont_attn_rect_tc");
  if (p.halves > 1) {
    attn_tc_combine_kernel<<<(unsigned)(total / 2), 256, 0, stream>>>(p.part, p.ctx, KV::WSCALE * p.W_out, p.Q, p.H,
                                                                       q_tiles, Bv);
    LTM_CHECK_LAUNCH("attn_tc_combine");
  }
  return 0;
}

// K, V, X: fp32 (KvTf32) or fp16 (KvF16) rows; see include/infltm.h
template <class KV>
static int cont_attn_rect_tc_impl(const float* q, const void* K, const void* V, int64_t ldkv, const void* X,
                                  const float* W, float W_out, float c_none, const int32_t* jb, const float* tb,
                                  float* ctx, float* scores_out, float* hist_part, float* part, int Bv, int Q, int N,
                                  int H, int d, void* stream) {
  const int halves = part != nullptr ? 2 : 1;
  const int NBk = N / halves;                        // basis functions per work item
  LTM_REQUIRE(q && K && V && X && W && ctx, "%s: null pointer", KV::NAME);
  LTM_REQUIRE(hist_part == nullptr || (jb && tb), "%s: histogram requested without edge tables", KV::NAME);
  LTM_REQUIRE(Bv > 0 && Bv <= 65535 && Q > 0 && H > 0 && H <= 65535 && ldkv % (KV::HALF ? 8 : 4) == 0 &&
                  ldkv >= (int64_t)H * d,
              "%s: bad shape", KV::NAME);
  LTM_REQUIRE(aligned16(q) && aligned16(ctx) && aligned16(part), "%s: 16-byte alignment", KV::NAME);
  CUtensorMap mK, mV, mX;
  const unsigned long long rows = (unsigned long long)Bv * N, hd = (unsigned long long)H * d;
  if constexpr (KV::HALF) {
    if (tma_encode_2d_f16(&mK, K, hd, rows, (unsigned long long)ldkv, (unsigned)NBk, "attn16 K")) return -1;
    if (tma_encode_2d_f16(&mV, V, hd, rows, (unsigned long long)ldkv, (unsigned)NBk, "attn16 V")) return -1;
    if (tma_encode_2d_f16(&mX, X, 64, (unsigned long long)N, 64, (unsigned)NBk, "attn16 X")) return -1;
  } else {
    const float *Kf = static_cast<const float*>(K), *Vf = static_cast<const float*>(V);
    const float* Xf = static_cast<const float*>(X);
    if (tma_encode_2d(&mK, Kf, hd, rows, (unsigned long long)ldkv, 32, (unsigned)NBk, 0, "attn K")) return -1;
    if (tma_encode_2d(&mV, Vf, hd, rows, (unsigned long long)ldkv, 32, (unsigned)NBk, 1, "attn V")) return -1;
    if (tma_encode_2d(&mX, Xf, 32, (unsigned long long)N, 32, 32, (unsigned)NBk, 1, "attn X")) return -1;
  }
  Params p{};
  p.q = q; p.W = W; p.tb = tb; p.jb = jb; p.W_out = W_out; p.c_none = c_none; p.ctx = ctx;
  p.scores_out = scores_out; p.hist_part = hist_part; p.Q = Q; p.H = H;
  p.halves = halves; p.NT = N; p.part = part;
  if (NBk == 256) return launch<256, KV>(mK, mV, mX, p, Bv, (cudaStream_t)stream);
  if (NBk == 128) return launch<128, KV>(mK, mV, mX, p, Bv, (cudaStream_t)stream);
  return launch<64, KV>(mK, mV, mX, p, Bv, (cudaStream_t)stream);
}

}  // namespace tc
}  // namespace ltm

extern "C" int ltm_attn_tc_supported(int N, int d) { return (d == 64 && (N == 64 || N == 128 || N == 256)) ? 1 : 0; }
extern "C" int ltm_attn_tc_split_supported(int N, int d) { return (d == 64 && N == 512) ? 1 : 0; }
extern "C" int64_t ltm_attn_tc_split_workspace_floats(int Bv, int Q, int H) {
  return (int64_t)Bv * H * ((Q + ltm::tc::QT - 1) / ltm::tc::QT) * 2 * ltm::tc::PART_ROWS * ltm::tc::QT;
}

extern "C" int ltm_cont_attn_rect_tc(const float* q, const float* K, const float* V, int64_t ldkv, const float* X,
                                     const float* W, float W_out, float c_none, const int32_t* jb, const float* tb,
                                     float* ctx, float* scores_out, float* hist_part, int Bv, int Q, int N, int H,
                                     int d, void* stream) {
  using namespace ltm;
  LTM_REQUIRE(ltm_attn_tc_supported(N, d), "cont_attn_rect_tc: unsupported num_basis=%d / head_size=%d", N, d);
  return tc::cont_attn_rect_tc_impl<tc::KvTf32>(q, K, V, ldkv, X, W, W_out, c_none, jb, tb, ctx, scores_out, hist_part,
                                                nullptr, Bv, Q, N, H, d, stream);
}

// num_basis 512: two work items per (query tile, head, video), merged by attn_tc_combine_kernel; the sticky
// histogram of the next call then comes from the stored scores (ltm_sticky_hist_rect_tiles), because the density of a
// basis needs the normaliser over BOTH halves.  scores_ws[Bv,H,Q,N] and part_ws (ltm_attn_tc_split_workspace_floats)
// are caller-provided workspaces.
extern "C" int ltm_cont_attn_rect_tc_split(const float* q, const float* K, const float* V, int64_t ldkv,
                                           const float* X, const float* W, float W_out, const int32_t* jb,
                                           const float* tb, float* ctx, float* scores_ws, float* part_ws,
                                           float* hist_part, int Bv, int Q, int N, int H, int d, void* stream) {
  using namespace ltm;
  LTM_REQUIRE(ltm_attn_tc_split_supported(N, d), "cont_attn_rect_tc_split: unsupported num_basis=%d / head_size=%d", N, d);
  LTM_REQUIRE(part_ws != nullptr && (hist_part == nullptr || scores_ws != nullptr),
              "cont_attn_rect_tc_split: workspaces missing");
  int rc = tc::cont_attn_rect_tc_impl<tc::KvTf32>(q, K, V, ldkv, X, W, W_out, 0.f, jb, tb, ctx, scores_ws, nullptr,
                                                  part_ws, Bv, Q, N, H, d, stream);
  if (rc || hist_part == nullptr) return rc;
  return ltm_sticky_hist_rect_tiles(scores_ws, jb, tb, hist_part, Bv, H, Q, N, stream);
}

extern "C" int ltm_cont_attn_rect_tc16(const float* q, const void* K, const void* V, int64_t ldkv, const void* X,
                                       const float* W, float W_out, float c_none, const int32_t* jb, const float* tb,
                                       float* ctx, float* scores_out, float* hist_part, int Bv, int Q, int N, int H,
                                       int d, void* stream) {
  using namespace ltm;
  LTM_REQUIRE(ltm_attn_tc_supported(N, d), "cont_attn_rect_tc16: unsupported num_basis=%d / head_size=%d", N, d);
  return tc::cont_attn_rect_tc_impl<tc::KvF16>(q, K, V, ldkv, X, W, W_out, c_none, jb, tb, ctx, scores_out, hist_part,
                                               nullptr, Bv, Q, N, H, d, stream);
}

extern "C" int ltm_cont_attn_rect_tc16_split(const float* q, const void* K, const void* V, int64_t ldkv,
                                             const void* X, const float* W, float W_out, const int32_t* jb,
                                             const float* tb, float* ctx, float* scores_ws, float* part_ws,
                                             float* hist_part, int Bv, int Q, int N, int H, int d, void* stream) {
  using namespace ltm;
  LTM_REQUIRE(ltm_attn_tc_split_supported(N, d), "cont_attn_rect_tc16_split: unsupported num_basis=%d / head_size=%d",
              N, d);
  LTM_REQUIRE(part_ws != nullptr && (hist_part == nullptr || scores_ws != nullptr),
              "cont_attn_rect_tc16_split: workspaces missing");
  int rc = tc::cont_attn_rect_tc_impl<tc::KvF16>(q, K, V, ldkv, X, W, W_out, 0.f, jb, tb, ctx, scores_ws, nullptr,
                                                 part_ws, Bv, Q, N, H, d, stream);
  if (rc || hist_part == nullptr) return rc;
  return ltm_sticky_hist_rect_tiles(scores_ws, jb, tb, hist_part, Bv, H, Q, N, stream);
}
