// Batched fp32-in / fp32-out GEMM on the 5th-generation tensor cores of sm_100a.
//
//   C[b] (M x Nc) = A[b] (M x K) * B[b] (K x Nc) (+ bias)         tcgen05.mma kind::tf32
//
// * operands stay fp32 in HBM; TMA (cp.async.bulk.tensor, SWIZZLE_128B) drops 128x32 / BNx32 tiles
//   into shared memory, the tensor core reads them as TF32, the accumulator lives in TMEM (fp32) and
//   comes back through tcgen05.ld for the bias/store epilogue.
// * both operand major-nesses are supported (K-major rows of 32 floats, or MN-major slabs of
//   [32 k][32 mn]); B may be the row-concatenation of two tensors (the Gaussian variant regresses
//   [re-sampled memory ; new chunk] without materialising the concatenation,
//   long_term_attention.py:249-250).
// * precision 3 = split-TF32: the tensor core truncates fp32 -> tf32 (hi = tf32(x) is the loaded tile itself);
//   8 warps write lo = x - hi into two alternating buffers and three MMAs (hi*hi + lo*hi + hi*lo) reproduce
//   fp32-grade products.  Needed for the Gaussian variant whose RBF design values reach 80 with heavy
//   cancellation (single-pass TF32 -> 1e-2 error).
// * ab_fp16: both operands IEEE fp16 (64 K-elements per 128-byte row, kind::f16, K = 16 per MMA), same pipeline.
//
// Persistent, warp-specialised: warp 0 = TMA producer, warp 1 = TMEM owner + MMA issuer, warps 2-9 =
// epilogue (TMEM lane quarter = warp_id % 4, two warps per quarter), warps 10-17 = operand splitter (precision 3
// only); two TMEM accumulators so the epilogue of one tile overlaps the MMAs of the next.
#include <cuda.h>
#include <cudaTypedefs.h>
#include <cuda_fp16.h>

#include "common.cuh"
#include "tcgen05.cuh"

namespace ltm {

int gemm_simt_launch(const ltm_gemm_args& g, cudaStream_t stream);

constexpr int BM = 128;
constexpr int BK = 32;                       // 32 fp32 = 128 B = one SWIZZLE_128B row
constexpr int UMMA_K = 8;                    // 32 B of K per tcgen05.mma for tf32
constexpr int A_BYTES = BM * BK * 4;         // 16 KB
constexpr int SLAB_BYTES = 32 * BK * 4;      // MN-major slab: 32 k-rows x 128 B

struct GemmDev {
  float* C;
  const float* bias;
  long long ldc, strideC;
  int M, Nc, K, K1, batch;
  int a_kmajor, b_kmajor;
  int a_batched, b_batched, b2_batched, has_b2;
  unsigned mn_layout, mn_lbo, mn_sbo, mn_kadv;
  float* CT;
  int ct_cols, ct_group;
  int c_group;
  long long c_group_stride, bias_stride;
  int ab_half;                              // operands are fp16 (kind::f16, 64 K-elements per 128-byte row)
  int round_tf32;                           // round stored row-major results to the tf32 grid
  int c_vec;                                // row-major fp32 stores may be 128-bit (alignment checked on the host)
  int c_vec8;                               // fp16 stores may be 128-bit: 8 halves (alignment checked on the host)
  int a_group;                              // two-level row mapping of A (0 = off): tile rows span 128 / a_group groups
  int c_half;                               // C is fp16 storage (row-major path only)
  void* C_lo;                               // fp16 output only: second array for the residual x - float(half(x))
  int max_ctas;                             // bound of the persistent grid (0 = one CTA per SM)
  const int32_t* n_ext;                     // EXT instances: per-batch column bound (NULL = Nc) ...
  const int32_t* k_ext;                     // ... and K bound, a multiple of the 64-element fp16 k-block (NULL = K)
};

// Work item -> tile origin: items are tiles, n fastest.
template <int BN_>
__device__ __forceinline__ void decode_work(int w, int tiles_n, int tiles_m, int& n0, int& m0, int& bz) {
  n0 = (w % tiles_n) * BN_;
  m0 = ((w / tiles_n) % tiles_m) * 128;
  bz = w / (tiles_n * tiles_m);
}
// k-blocks of a tile of batch bz: all of them, or (EXT with k_ext) k_ext[bz] / 64 of them (fp16 k-blocks)
template <bool EXT>
__device__ __forceinline__ int tile_kb(const GemmDev& g, int bz, int num_kb) {
  if (!EXT || g.k_ext == nullptr) return num_kb;
  const int kb = __ldg(g.k_ext + bz) / 64;
  return kb < num_kb ? kb : num_kb;
}
// First work item >= w of this CTA's static list that has work: without EXT, w itself; with EXT, tiles whose first
// column lies at or past n_ext[bz], or whose batch runs no k-block, are skipped.  Every role walks the list through
// this function, so producer, MMA issuer and epilogue agree on the tiles they skip.
template <bool EXT, int BN_>
__device__ __forceinline__ int next_work(const GemmDev& g, int w, int stride, int num_work, int tiles_n, int tiles_m,
                                         int num_kb) {
  if (EXT) {
    for (; w < num_work; w += stride) {
      int n0, m0, bz;
      decode_work<BN_>(w, tiles_n, tiles_m, n0, m0, bz);
      if ((g.n_ext == nullptr || n0 < __ldg(g.n_ext + bz)) && tile_kb<true>(g, bz, num_kb) > 0) break;
    }
  }
  return w;
}
// MN-major descriptor parameters.  For 32-bit (tf32) MN-major operands the only legal canonical layout is
// the 128-byte swizzle with 32-byte atoms (TMA: SWIZZLE_128B_ATOM_32B): atoms of [4 k][32 mn], i.e. the
// K groups are 4 rows = 512 B apart (SBO), the 32-wide MN atoms one slab = 4096 B apart (LBO), and one
// MMA (K = 8) advances two K groups = 1024 B.  fp16 operands use other values (set on the host per call).
struct MnDesc { uint32_t layout, lbo, sbo, kadv; };
// K-major tile [rows][32 fp32], SWIZZLE_128B: 8-row groups 1024 B apart (SBO); K advances 32 B inside the
// swizzle row.  MN-major tile [mn/32 slabs][32 k][32 fp32]: see MnDesc.
__device__ __forceinline__ uint64_t operand_desc(uint32_t tile, int kmajor, int k, const MnDesc& mn) {
  return kmajor ? umma_desc(tile + k * (UMMA_K * 4), 16, 1024, 2u)
                : umma_desc(tile + k * mn.kadv, mn.lbo, mn.sbo, mn.layout);
}
// The same descriptor as (low word at address 0, high word, low-word step per MMA): low word of an operand at
// shared address `a` (a < 256 KB, 16-byte aligned) after k MMAs = lo0 + (a >> 4) + k * kstep.
struct DescWords { uint32_t lo0, hi, kstep; };
__device__ __forceinline__ DescWords operand_desc_words(int kmajor, const MnDesc& mn) {
  const uint64_t d = operand_desc(0u, kmajor, 0, mn);
  DescWords w;
  w.lo0 = (uint32_t)d;
  w.hi = (uint32_t)(d >> 32);
  w.kstep = (kmajor ? (uint32_t)(UMMA_K * 4) : mn.kadv) >> 4;
  return w;
}

// Epilogue: 8 warps (two per TMEM lane quarter, each owning half of the tile's columns) drain the accumulator in
// chunks of 32 columns: tcgen05.ld.x32 -> 8 x STS.128 into the warp's [32 rows][32 floats] staging tile (16-byte
// chunks XOR-swizzled with the row, so neither side has bank conflicts and no padding is needed) -> 8 x (LDS.128,
// + bias, STG.128) with a quarter-warp per row, i.e. every store instruction writes four full 128-byte lines.
// Row offsets (the two-level mapping needs a division) and the tile's bias values are computed / fetched once per
// tile, before the wait for the accumulator.  The first version did that arithmetic per store on 4 warps:
// ~28 k cycles per 128 x 256 tile, 2.3x the tile's MMA time, and that -- not shared-memory bandwidth -- was what
// held the kernel at 47 % tensor-pipe activity.
constexpr int EPI_WARPS = 8;                           // each TMEM lane quarter is served by EPI_WARPS / 4 warps
constexpr int EPI_SPLIT = EPI_WARPS / 4;
constexpr int EPI_THREADS = EPI_WARPS * 32;
constexpr int EPI_COLS = 32;
constexpr int STG_WARP_FLOATS = 32 * EPI_COLS;
constexpr int STG_BYTES = EPI_WARPS * STG_WARP_FLOATS * 4;
constexpr int ROLE_THREADS = 64 + EPI_THREADS;                // TMA warp + MMA warp + epilogue warps
// Register cap: the kernel needs one CTA per SM, but frame pooling of the next chunk runs beside it on a second
// stream (9.7 k registers per pooling CTA); 320 threads x 96 registers leave room for three of them.
constexpr int GEMM_MAX_REGS = 96;

// Drains one 128-row accumulator tile.  `ew` = epilogue warp 0..7 (its CTA warp id & 3 must be ew & 3: a warp can
// only read its own TMEM lane quarter), `tmem_acc` = TMEM address of the tile's first column.
template <int BN, bool HOUT>
__device__ __forceinline__ void epilogue_tile(const GemmDev& g, uint32_t tmem_acc, int ew, int warp_quarter, int lane,
                                              float* stg, int m0, int n0, int bz, uint32_t tfull, uint32_t tfull_parity) {
  const int row0 = m0 + warp_quarter * 32;
  constexpr int WCOLS = BN / EPI_SPLIT;            // columns drained by this warp
  const int cbeg = (ew >> 2) * WCOLS;
  float* cbase_ptr = g.C + (size_t)bz * g.strideC;
  const float* bias = g.bias ? g.bias + (size_t)bz * g.bias_stride : nullptr;
  // rows this lane stores in the row-major path: 4 i + (lane >> 3); its 16-byte column chunk: lane & 7
  // (fp16 output: 8 rows per pass, four lanes per row, 8 columns = one 16-byte store per lane; passes i < 4)
  const int lrow = HOUT ? lane >> 2 : lane >> 3, lchunk = HOUT ? lane & 3 : lane & 7;
  constexpr int rstep = HOUT ? 8 : 4;
  size_t roff[8];
  bool rok[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int row = row0 + rstep * i + lrow;
    rok[i] = row < g.M;
    roff[i] = g.c_group > 0 ? (size_t)(row / g.c_group) * g.c_group_stride + (size_t)(row % g.c_group) * g.ldc
                            : (size_t)row * g.ldc;
  }
  // transposed path: this lane owns row (row0 + lane)
  const int trow = row0 + lane;
  float* tbase = nullptr;
  if (g.CT != nullptr && trow < g.M)
    tbase = g.CT + (size_t)bz * g.strideC + (size_t)(trow / g.ct_group) * g.ct_cols * g.ct_group + (trow % g.ct_group);
  //   row-major path: bvs[j] = bias of this lane's 4 columns in chunk j;
  //   transposed path: btr[j] = bias[n0 + cbeg + 32 j + lane], redistributed with shuffles.
  constexpr int NCH = WCOLS / EPI_COLS;
  float4 bvs[NCH];
  float btr[NCH];
#pragma unroll
  for (int j = 0; j < NCH; ++j) {
    bvs[j] = make_float4(0.f, 0.f, 0.f, 0.f);
    btr[j] = 0.f;
  }
  if (bias != nullptr) {
    if (g.CT != nullptr && n0 + cbeg < g.ct_cols) {                      // some chunks take the transposed path
#pragma unroll
      for (int j = 0; j < NCH; ++j) {
        const int col = n0 + cbeg + EPI_COLS * j + lane;
        if (col < g.Nc) btr[j] = __ldg(bias + col);
      }
    }
    if (g.CT == nullptr || n0 + cbeg + WCOLS > g.ct_cols) {             // some chunks take the row-major path
#pragma unroll
      for (int j = 0; j < NCH; ++j) {
        const int col = n0 + cbeg + EPI_COLS * j + 4 * lchunk;
        if (col + 0 < g.Nc) bvs[j].x = __ldg(bias + col + 0);
        if (col + 1 < g.Nc) bvs[j].y = __ldg(bias + col + 1);
        if (col + 2 < g.Nc) bvs[j].z = __ldg(bias + col + 2);
        if (col + 3 < g.Nc) bvs[j].w = __ldg(bias + col + 3);
      }
    }
  }
  mbar_wait(tfull, tfull_parity);
  tcgen05_fence_after();
#pragma unroll
  for (int j = 0; j < NCH; ++j) {
    const int c0 = cbeg + j * EPI_COLS;
    if (n0 + c0 >= g.Nc) break;                    // warp-uniform
    uint32_t r[32];
    const uint32_t taddr = tmem_acc + ((uint32_t)(warp_quarter * 32) << 16) + (uint32_t)c0;
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
    if (g.CT != nullptr && n0 + c0 < g.ct_cols) {
      // transposed store (keys per head): lanes are consecutive rows of one group -> 128-byte coalesced
      float* dst = tbase + (size_t)(n0 + c0) * g.ct_group;
#pragma unroll
      for (int i = 0; i < 32; ++i) {
        const float b = __shfl_sync(0xffffffffu, btr[j], i);             // all lanes take part
        if (tbase != nullptr) dst[(size_t)i * g.ct_group] = __uint_as_float(r[i]) + b;
      }
      continue;
    }
    // row-major store through the warp's staging tile: row `lane`, chunk q at position q ^ (lane & 7)
#pragma unroll
    for (int q = 0; q < 8; ++q)
      *reinterpret_cast<float4*>(stg + lane * EPI_COLS + ((q ^ (lane & 7)) << 2)) =
          make_float4(__uint_as_float(r[4 * q]), __uint_as_float(r[4 * q + 1]), __uint_as_float(r[4 * q + 2]),
                      __uint_as_float(r[4 * q + 3]));
    __syncwarp();
    if (HOUT) {
      // fp16 rows: lane -> (row 8 i + lane / 4, columns 8 (lane % 4) .. + 7): two staged 16-byte chunks -> one 16-byte
      // store of 8 halves (rows of 64 B per warp-wide store)
      const int col8 = n0 + c0 + 8 * lchunk;
      const bool vec8 = g.c_vec8 && (col8 + 7 < g.Nc);
      float bb[8];
#pragma unroll
      for (int t = 0; t < 8; ++t) bb[t] = (bias != nullptr && col8 + t < g.Nc) ? __ldg(bias + col8 + t) : 0.f;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int srow = 8 * i + lrow;
        const float4 v0 = *reinterpret_cast<const float4*>(stg + srow * EPI_COLS + (((2 * lchunk) ^ (srow & 7)) << 2));
        const float4 v1 = *reinterpret_cast<const float4*>(stg + srow * EPI_COLS + (((2 * lchunk + 1) ^ (srow & 7)) << 2));
        const float f[8] = {v0.x + bb[0], v0.y + bb[1], v0.z + bb[2], v0.w + bb[3],
                            v1.x + bb[4], v1.y + bb[5], v1.z + bb[6], v1.w + bb[7]};
        if (rok[i]) {
          __half* dst = reinterpret_cast<__half*>(g.C) + (size_t)bz * g.strideC + roff[i] + (col8 - (g.CT != nullptr ? g.ct_cols : 0));
          __half* dlo = g.C_lo ? reinterpret_cast<__half*>(g.C_lo) + (dst - reinterpret_cast<__half*>(g.C)) : nullptr;
          if (vec8) {
            uint4 pk;
            __half2 h[4];
#pragma unroll
            for (int t = 0; t < 4; ++t) h[t] = __floats2half2_rn(f[2 * t], f[2 * t + 1]);
            pk.x = *reinterpret_cast<const uint32_t*>(&h[0]); pk.y = *reinterpret_cast<const uint32_t*>(&h[1]);
            pk.z = *reinterpret_cast<const uint32_t*>(&h[2]); pk.w = *reinterpret_cast<const uint32_t*>(&h[3]);
            *reinterpret_cast<uint4*>(dst) = pk;
            if (dlo != nullptr) {                    // residual term: x ~ hi + lo, 22 significant bits
              __half2 l[4];
#pragma unroll
              for (int t = 0; t < 4; ++t) {
                const float2 hf = __half22float2(h[t]);
                l[t] = __floats2half2_rn(f[2 * t] - hf.x, f[2 * t + 1] - hf.y);
              }
              pk.x = *reinterpret_cast<const uint32_t*>(&l[0]); pk.y = *reinterpret_cast<const uint32_t*>(&l[1]);
              pk.z = *reinterpret_cast<const uint32_t*>(&l[2]); pk.w = *reinterpret_cast<const uint32_t*>(&l[3]);
              *reinterpret_cast<uint4*>(dlo) = pk;
            }
          } else {
#pragma unroll
            for (int t = 0; t < 8; ++t)
              if (col8 + t < g.Nc) {
                const __half hh = __float2half_rn(f[t]);
                dst[t] = hh;
                if (dlo != nullptr) dlo[t] = __float2half_rn(f[t] - __half2float(hh));
              }
          }
        }
      }
      __syncwarp();
      continue;
    }
    const int col = n0 + c0 + 4 * lchunk;
    const float4 bv = bvs[j];
    const int ccol = col - (g.CT != nullptr ? g.ct_cols : 0);
    const bool vec = g.c_vec && (col + 3 < g.Nc);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int srow = 4 * i + lrow;
      float4 v = *reinterpret_cast<const float4*>(stg + srow * EPI_COLS + ((lchunk ^ (srow & 7)) << 2));
      v.x += bv.x; v.y += bv.y; v.z += bv.z; v.w += bv.w;
      if (g.round_tf32) v = make_float4(tf32_rna(v.x), tf32_rna(v.y), tf32_rna(v.z), tf32_rna(v.w));
      if (rok[i]) {
        float* dst = cbase_ptr + roff[i] + ccol;
        if (vec) {
          *reinterpret_cast<float4*>(dst) = v;
        } else {
          if (col + 0 < g.Nc) dst[0] = v.x;
          if (col + 1 < g.Nc) dst[1] = v.y;
          if (col + 2 < g.Nc) dst[2] = v.z;
          if (col + 3 < g.Nc) dst[3] = v.w;
        }
      }
    }
    __syncwarp();
  }
}

template <int BN, int STAGES, bool SPLIT>
struct Cfg {
  static constexpr int B_BYTES = BN * BK * 4;
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;        // TMA landing slot ("hi" operands are used in place)
  static constexpr int LO_BYTES = SPLIT ? 2 * STAGE_BYTES : 0; // two buffers of lo = x - tf32(x) (precision 3)
  static constexpr int RING_BYTES = STAGES * STAGE_BYTES + LO_BYTES;
  static constexpr int BAR_BYTES = 256;
  static constexpr int SMEM_BYTES = RING_BYTES + STG_BYTES + BAR_BYTES + 1024;   // + 1024 B alignment slack
  static constexpr int TMEM_COLS = 2 * BN;                     // two accumulator buffers (256 or 512 columns)
  static constexpr int SPLIT_THREADS = 256;                    // 8 splitter warps (precision 3)
  static constexpr int THREADS = SPLIT ? ROLE_THREADS + SPLIT_THREADS : ROLE_THREADS;
  static_assert(TMEM_COLS == 256 || TMEM_COLS == 512, "TMEM allocation must be a power of two <= 512");
};

// Persistent kernel: grid = min(#tiles, #SMs); every role walks the same static tile sequence
// t = blockIdx.x, blockIdx.x + gridDim.x, ...  (tile -> (batch, m, n), n fastest so that CTAs running at the
// same time share the A rows).  The smem ring and its phases run continuously across tiles; the accumulator is
// double-buffered in TMEM so the epilogue of tile i drains while the MMAs of tile i+1 run.
//   warp 0      TMA producer (one lane)
//   warp 1      TMEM owner + tcgen05.mma issuer (one lane)
//   warps 2-9   epilogue (see epilogue_tile)
//   warps 10-17 (precision 3 only) operand splitter hi/lo
//   EXT: per-batch extents (n_ext / k_ext, see next_work and tile_kb)
template <int BN, int STAGES, bool SPLIT, bool HOUT, bool EXT>
__global__ void __maxnreg__(GEMM_MAX_REGS)
gemm_tf32_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB,
                 const __grid_constant__ CUtensorMap mapB2, const GemmDev g) {
  using C_ = Cfg<BN, STAGES, SPLIT>;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;     // SWIZZLE_128B wants 1024 B alignment
  uint8_t* smem_al = smem_raw + (smem_base - smem_u32(smem_raw));
  float* staging = reinterpret_cast<float*>(smem_al + C_::RING_BYTES);
  const uint32_t bars = smem_base + C_::RING_BYTES + STG_BYTES;
  auto full_bar = [&](int s) { return bars + 8u * s; };
  auto empty_bar = [&](int s) { return bars + 8u * (STAGES + s); };
  auto split_bar = [&](int s) { return bars + 8u * (2 * STAGES + s); };
  auto tfull_bar = [&](int b) { return bars + 8u * (3 * STAGES + b); };
  auto tempty_bar = [&](int b) { return bars + 8u * (3 * STAGES + 2 + b); };
  auto lofree_bar = [&](uint32_t b) { return bars + 8u * (3 * STAGES + 4 + b); };
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem_al + C_::RING_BYTES + STG_BYTES + 8 * (3 * STAGES + 6));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int bke = g.ab_half ? 2 * BK : BK;        // K-elements per 128-byte swizzle row
  const int num_kb = (g.K + bke - 1) / bke;
  const int tiles_n = (g.Nc + BN - 1) / BN, tiles_m = (g.M + BM - 1) / BM;
  // static work list shared by all roles (see decode_work)
  const int w_first = blockIdx.x, w_stride = gridDim.x;
  const int num_work = tiles_n * tiles_m * g.batch;

  if (threadIdx.x == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&mapA)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&mapB)) : "memory");
    if (g.has_b2) asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&mapB2)) : "memory");
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), 1);        // tcgen05.commit once the MMAs have read the slot
      mbar_init(split_bar(s), C_::SPLIT_THREADS);   // every splitter thread arrives after its proxy fence
    }
    mbar_init(lofree_bar(0), 1);         // MMAs of a k-block done with their lo buffer (two, alternating)
    mbar_init(lofree_bar(1), 1);
    for (int b = 0; b < 2; ++b) {
      mbar_init(tfull_bar(b), 1);        // tcgen05.commit of the last MMA of a tile
      mbar_init(tempty_bar(b), EPI_THREADS);   // every epilogue thread after its last tcgen05.ld of the tile
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                 "r"((uint32_t)C_::TMEM_COLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer
    if (lane == 0) {
      uint32_t it = 0;
      for (int w = next_work<EXT, BN>(g, w_first, w_stride, num_work, tiles_n, tiles_m, num_kb); w < num_work;
           w = next_work<EXT, BN>(g, w + w_stride, w_stride, num_work, tiles_n, tiles_m, num_kb)) {
        int n0, m0, bz;
        decode_work<BN>(w, tiles_n, tiles_m, n0, m0, bz);
        const int za = g.a_batched ? bz : 0;
        const int nkb = tile_kb<EXT>(g, bz, num_kb);
        for (int kb = 0; kb < nkb; ++kb, ++it) {
          const int s = it % STAGES;
          const uint32_t ph = (it / STAGES) & 1u;
          mbar_wait(empty_bar(s), ph ^ 1u);
          mbar_arrive_expect_tx(full_bar(s), A_BYTES + C_::B_BYTES);
          const uint32_t sa = smem_base + s * C_::STAGE_BYTES;
          const uint32_t sb = sa + A_BYTES;
          const int k0 = kb * bke;
          if (g.a_group > 0) {
            // grouped rows: the tensor map is {K, a_group rows, groups}; one box covers 128 flat rows
            tma_load_3d(&mapA, sa, full_bar(s), k0, g.a_group > BM ? m0 % g.a_group : 0, m0 / g.a_group);
          } else if (g.a_kmajor) {
            tma_load_3d(&mapA, sa, full_bar(s), k0, m0, za);
          } else {
#pragma unroll
            for (int i = 0; i < BM / 32; ++i)
              tma_load_3d(&mapA, sa + i * SLAB_BYTES, full_bar(s), m0 + 32 * i, k0, za);
          }
          const bool seg2 = g.has_b2 && (k0 >= g.K1);
          const CUtensorMap* mb = seg2 ? &mapB2 : &mapB;
          const int kk = seg2 ? k0 - g.K1 : k0;
          const int zb = seg2 ? (g.b2_batched ? bz : 0) : (g.b_batched ? bz : 0);
          if (g.b_kmajor) {
            tma_load_3d(mb, sb, full_bar(s), kk, n0, zb);
          } else if (g.ab_half) {
            // 16-bit MN-major: slabs of [64 k rows][64 n halves = 128 B], one per 64 columns of the tile
#pragma unroll
            for (int i = 0; i < BN / 64; ++i)
              tma_load_3d(mb, sb + i * (64 * 128), full_bar(s), n0 + 64 * i, kk, zb);
          } else {
#pragma unroll
            for (int i = 0; i < BN / 32; ++i)
              tma_load_3d(mb, sb + i * SLAB_BYTES, full_bar(s), n0 + 32 * i, kk, zb);
          }
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer
    if (lane == 0) {
      // instruction descriptor: D=f32 [4,6)=1, A=tf32 [7,10)=2, B=tf32 [10,13)=2, a_major bit15,
      // b_major bit16 (1 = MN-major), N>>3 [17,23), M>>4 [24,29)
      const uint32_t fmt = g.ab_half ? 0u : 2u;         // operand format: 0 = f16 (kind::f16), 2 = tf32
      const uint32_t idesc = (1u << 4) | (fmt << 7) | (fmt << 10) | ((g.a_kmajor ? 0u : 1u) << 15) |
                             ((g.b_kmajor ? 0u : 1u) << 16) | ((uint32_t)(BN >> 3) << 17) |
                             ((uint32_t)(BM >> 4) << 24);
      const MnDesc mn{g.mn_layout, g.mn_lbo, g.mn_sbo, g.mn_kadv};
      const DescWords wa = operand_desc_words(g.a_kmajor, mn), wb = operand_desc_words(g.b_kmajor, mn);
      const uint32_t da0 = wa.lo0 + ((smem_base & 0x3FFFFu) >> 4), db0 = wb.lo0 + (((smem_base + A_BYTES) & 0x3FFFFu) >> 4);
      const uint32_t dal0 = da0 + STAGES * (C_::STAGE_BYTES >> 4), dbl0 = db0 + STAGES * (C_::STAGE_BYTES >> 4);
      uint32_t it = 0, tc = 0;
      for (int w = next_work<EXT, BN>(g, w_first, w_stride, num_work, tiles_n, tiles_m, num_kb); w < num_work;
           w = next_work<EXT, BN>(g, w + w_stride, w_stride, num_work, tiles_n, tiles_m, num_kb), ++tc) {
        int n0, m0, bz;
        decode_work<BN>(w, tiles_n, tiles_m, n0, m0, bz);
        const int nkb = tile_kb<EXT>(g, bz, num_kb);
        const uint32_t buf = tc & 1u, tph = (tc >> 1) & 1u;
        mbar_wait(tempty_bar(buf), tph ^ 1u);                 // epilogue has drained this accumulator
        tcgen05_fence_after();
        const uint32_t tmem_acc = tmem_base + buf * BN;
        for (int kb = 0; kb < nkb; ++kb, ++it) {
          const int s = it % STAGES;
          const uint32_t ph = (it / STAGES) & 1u;
          mbar_wait(SPLIT ? split_bar(s) : full_bar(s), ph);
          tcgen05_fence_after();
          uint32_t da = da0 + s * (C_::STAGE_BYTES >> 4), db = db0 + s * (C_::STAGE_BYTES >> 4);
          const uint32_t lob = (it & 1u) * (C_::STAGE_BYTES >> 4);     // lo buffer [A_lo | B_lo] of this k-block
          uint32_t dal = dal0 + lob, dbl = dbl0 + lob;
#pragma unroll
          for (int k = 0; k < BK / UMMA_K; ++k) {
            if (g.ab_half) tcgen05_mma_f16(tmem_acc, da, wa.hi, db, wb.hi, idesc, (kb | k) != 0 ? 1u : 0u);
            else tcgen05_mma_tf32(tmem_acc, da, wa.hi, db, wb.hi, idesc, (kb | k) != 0 ? 1u : 0u);
            if (SPLIT) {
              tcgen05_mma_tf32(tmem_acc, dal, wa.hi, db, wb.hi, idesc, 1u);
              tcgen05_mma_tf32(tmem_acc, da, wa.hi, dbl, wb.hi, idesc, 1u);
              dal += wa.kstep; dbl += wb.kstep;
            }
            da += wa.kstep; db += wb.kstep;
          }
          if (SPLIT) tcgen05_commit(lofree_bar(it & 1u));  // the splitter may overwrite this lo buffer
          tcgen05_commit(empty_bar(s));            // frees the stage once these MMAs have read it
        }
        tcgen05_commit(tfull_bar(buf));          // accumulator of this tile complete
      }
    }
    __syncwarp();
  } else if (warp < 2 + EPI_WARPS) {
    // ------------------------------------------------------------------ epilogue warps
    const int ew = warp - 2;
    float* stg = staging + ew * STG_WARP_FLOATS;
    uint32_t tc = 0;
    for (int w = next_work<EXT, BN>(g, w_first, w_stride, num_work, tiles_n, tiles_m, num_kb); w < num_work;
         w = next_work<EXT, BN>(g, w + w_stride, w_stride, num_work, tiles_n, tiles_m, num_kb), ++tc) {
      int n0, m0, bz;
      decode_work<BN>(w, tiles_n, tiles_m, n0, m0, bz);
      const uint32_t buf = tc & 1u, tph = (tc >> 1) & 1u;
      epilogue_tile<BN, HOUT>(g, tmem_base + buf * BN, ew, warp & 3, lane, stg, m0, n0, bz, tfull_bar(buf), tph);
      tcgen05_fence_before();
      mbar_arrive(tempty_bar(buf));              // EPI_THREADS arrivals hand the accumulator back to the MMA warp
    }
  } else {
    // ------------------------------------------------------------------ operand splitter (precision 3)
    if (SPLIT) {
      const int et = threadIdx.x - ROLE_THREADS;  // 0..SPLIT_THREADS-1
      constexpr int NV = (A_BYTES + C_::B_BYTES) / 16;      // float4 count of [A | B]
      uint32_t it = 0;
      for (int w = next_work<EXT, BN>(g, w_first, w_stride, num_work, tiles_n, tiles_m, num_kb); w < num_work;
           w = next_work<EXT, BN>(g, w + w_stride, w_stride, num_work, tiles_n, tiles_m, num_kb)) {
        int n0, m0, bz;
        decode_work<BN>(w, tiles_n, tiles_m, n0, m0, bz);
        const int nkb = tile_kb<EXT>(g, bz, num_kb);
        for (int kb = 0; kb < nkb; ++kb, ++it) {
          const int s = it % STAGES;
          const uint32_t ph = (it / STAGES) & 1u;
          mbar_wait(full_bar(s), ph);
          mbar_wait(lofree_bar(it & 1u), ((it >> 1) & 1u) ^ 1u);   // MMAs of k-block it - 2 have consumed this lo buffer
          const float4* hi = reinterpret_cast<const float4*>(smem_al + s * C_::STAGE_BYTES);
          float4* lo = reinterpret_cast<float4*>(smem_al + (STAGES + (it & 1u)) * C_::STAGE_BYTES);
#pragma unroll 4
          for (int f = et; f < NV; f += C_::SPLIT_THREADS) {
            const float4 x = hi[f];
            float4 h, l;
            h.x = __uint_as_float(__float_as_uint(x.x) & 0xFFFFE000u);
            h.y = __uint_as_float(__float_as_uint(x.y) & 0xFFFFE000u);
            h.z = __uint_as_float(__float_as_uint(x.z) & 0xFFFFE000u);
            h.w = __uint_as_float(__float_as_uint(x.w) & 0xFFFFE000u);
            l.x = x.x - h.x; l.y = x.y - h.y; l.z = x.z - h.z; l.w = x.w - h.w;
            // `hi` stays as loaded: the tensor core itself truncates fp32 -> tf32 (measured on B200: rewriting
            // the masked value gives bit-identical products)
            lo[f] = l;
          }
          asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic writes -> async proxy (UMMA)
          mbar_arrive(split_bar(s));
        }
      }
    }
  }

  tcgen05_fence_before();
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)C_::TMEM_COLS)
                 : "memory");
  }
}

// ------------------------------------------------------------------------------------------ host
static PFN_cuTensorMapEncodeTiled_v12000 g_encode = nullptr;
// MN-major tf32 operands: UMMA descriptor parameters (see MnDesc); their TMA maps use SWIZZLE_128B_ATOM_32B
constexpr MnDesc MN_TF32 = {1u, (uint32_t)SLAB_BYTES, 512u, 1024u};

static int resolve_encode() {
  if (g_encode) return 0;
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult qres;
  cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
  LTM_REQUIRE(e == cudaSuccess && fn != nullptr && qres == cudaDriverEntryPointSuccess,
              "gemm: cuTensorMapEncodeTiled unavailable (%s)", cudaGetErrorString(e));
  g_encode = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(fn);
  return 0;
}

// rows x K operand.  kmajor: memory [rows][K] -> dims {K, rows, batch}, box {32, box_rows, 1};
// otherwise memory [K][rows] -> dims {rows, K, batch}, box {32, 32, 1}.
static int encode_operand(CUtensorMap* map, const float* base, int rows, int K, long long ld, long long bstride,
                          int batch, int kmajor, int box_rows, const char* what, int half = 0) {
  if (half) {
    // fp16 operand.  K-major: memory [rows][K] halves -> dims {K, rows, batch}, box {64, box_rows, 1};
    // MN-major (B only): memory [K][rows] halves -> dims {rows, K, batch}, box {64, 64, 1} (one 8 KB slab per load)
    const long long inner = kmajor ? K : rows, outer = kmajor ? rows : K;
    LTM_REQUIRE(aligned16(base) && ld % 8 == 0 && ld >= inner && bstride % 8 == 0,
                "gemm: fp16 %s needs a 16-byte aligned base and pitches that are multiples of 8 elements", what);
    const int nbh = (bstride == 0) ? 1 : batch;
    cuuint64_t dims[3] = {(cuuint64_t)inner, (cuuint64_t)outer, (cuuint64_t)nbh};
    cuuint64_t strides[2] = {(cuuint64_t)ld * 2ull, (cuuint64_t)((bstride == 0 ? ld * outer : bstride) * 2ll)};
    cuuint32_t box[3] = {64u, (cuuint32_t)(kmajor ? box_rows : 64), 1u};
    cuuint32_t estr[3] = {1u, 1u, 1u};
    CUresult r = g_encode(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, const_cast<float*>(base), dims, strides, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    LTM_REQUIRE(r == CUDA_SUCCESS, "gemm: cuTensorMapEncodeTiled(%s, fp16) failed with CUresult %d", what, (int)r);
    return 0;
  }
  LTM_REQUIRE(aligned16(base), "gemm: %s base pointer must be 16-byte aligned", what);
  LTM_REQUIRE(ld % 4 == 0 && ld > 0, "gemm: %s leading dimension %lld must be a positive multiple of 4", what, ld);
  LTM_REQUIRE(bstride % 4 == 0, "gemm: %s batch stride %lld must be a multiple of 4", what, bstride);
  const int nb = (bstride == 0) ? 1 : batch;
  const long long inner = kmajor ? K : rows, outer = kmajor ? rows : K;
  LTM_REQUIRE(ld >= inner, "gemm: %s leading dimension %lld < inner extent %lld", what, ld, inner);
  cuuint64_t dims[3] = {(cuuint64_t)inner, (cuuint64_t)outer, (cuuint64_t)nb};
  cuuint64_t strides[2] = {(cuuint64_t)ld * 4ull, (cuuint64_t)((bstride == 0 ? ld * outer : bstride) * 4ll)};
  cuuint32_t box[3] = {32u, (cuuint32_t)(kmajor ? box_rows : 32), 1u};
  cuuint32_t estr[3] = {1u, 1u, 1u};
  CUresult r = g_encode(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(base), dims, strides, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE,
                        kmajor ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B,
                        CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  LTM_REQUIRE(r == CUDA_SUCCESS, "gemm: cuTensorMapEncodeTiled(%s) failed with CUresult %d", what, (int)r);
  return 0;
}

int tma_encode_2d(CUtensorMap* map, const float* base, unsigned long long inner, unsigned long long outer,
                  unsigned long long pitch_elems, unsigned box_inner, unsigned box_outer, int swizzle32b_atom,
                  const char* what) {
  if (resolve_encode()) return -1;
  LTM_REQUIRE(aligned16(base) && pitch_elems % 4 == 0 && pitch_elems >= inner, "%s: tensor map needs a 16-byte aligned base and pitch", what);
  LTM_REQUIRE(box_inner * 4 == 128 && box_outer >= 1 && box_outer <= 256, "%s: bad TMA box", what);
  cuuint64_t dims[2] = {(cuuint64_t)inner, (cuuint64_t)outer};
  cuuint64_t strides[1] = {(cuuint64_t)pitch_elems * 4ull};
  cuuint32_t box[2] = {box_inner, box_outer};
  cuuint32_t estr[2] = {1u, 1u};
  CUresult r = g_encode(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), dims, strides, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE,
                        swizzle32b_atom ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B : CU_TENSOR_MAP_SWIZZLE_128B,
                        CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  LTM_REQUIRE(r == CUDA_SUCCESS, "%s: cuTensorMapEncodeTiled failed with CUresult %d", what, (int)r);
  return 0;
}

int tma_encode_2d_f16(CUtensorMap* map, const void* base, unsigned long long inner, unsigned long long outer,
                      unsigned long long pitch_elems, unsigned box_outer, const char* what) {
  if (resolve_encode()) return -1;
  LTM_REQUIRE(aligned16(base) && pitch_elems % 8 == 0 && pitch_elems >= inner && box_outer >= 1 && box_outer <= 256,
              "%s: fp16 tensor map needs a 16-byte aligned base, a pitch that is a multiple of 8 halves, box <= 256", what);
  cuuint64_t dims[2] = {(cuuint64_t)inner, (cuuint64_t)outer};
  cuuint64_t strides[1] = {(cuuint64_t)pitch_elems * 2ull};
  cuuint32_t box[2] = {64u, box_outer};
  cuuint32_t estr[2] = {1u, 1u};
  CUresult r = g_encode(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  LTM_REQUIRE(r == CUDA_SUCCESS, "%s: cuTensorMapEncodeTiled failed with CUresult %d", what, (int)r);
  return 0;
}

template <int BN, int STAGES, bool SPLIT, bool HOUT = false, bool EXT = false>
static int launch_cfg(const CUtensorMap& mA, const CUtensorMap& mB, const CUtensorMap& mB2, const GemmDev& d,
                      int batch, cudaStream_t stream) {
  using C_ = Cfg<BN, STAGES, SPLIT>;
  static PerDevice pd = {};
  int num_sms = 0;
  if (int rc = kernel_setup(gemm_tf32_kernel<BN, STAGES, SPLIT, HOUT, EXT>, (size_t)C_::SMEM_BYTES, pd, &num_sms))
    return rc;
  const long long tiles = (long long)((d.Nc + BN - 1) / BN) * ((d.M + BM - 1) / BM) * batch;
  LTM_REQUIRE(tiles < (1ll << 31), "gemm: too many tiles");
  unsigned grid = (unsigned)(tiles < num_sms ? tiles : num_sms);     // persistent: one CTA per SM
  if (d.max_ctas > 0 && (unsigned)d.max_ctas < grid) grid = (unsigned)d.max_ctas;   // ... or fewer (ltm_gemm_args.max_ctas)
  gemm_tf32_kernel<BN, STAGES, SPLIT, HOUT, EXT><<<grid, C_::THREADS, C_::SMEM_BYTES, stream>>>(mA, mB, mB2, d);
  LTM_CHECK_LAUNCH("gemm(tcgen05)");
  return 0;
}

static int gemm_tcgen05_launch(const ltm_gemm_args& a, cudaStream_t stream, const int32_t* n_ext = nullptr,
                               const int32_t* k_ext = nullptr) {
  if (resolve_encode()) return -1;
  const bool two = a.B2 != nullptr && a.K1 < a.K;
  const int half = a.ab_fp16 ? 1 : 0;
  const int bke = half ? 2 * BK : BK;
  LTM_REQUIRE(!two || (a.K1 > 0 && a.K1 % bke == 0), "gemm: K1=%d must be a positive multiple of %d", a.K1, bke);
  LTM_REQUIRE(!half || (a.precision == 1 && a.a_kmajor), "gemm: fp16 operands need precision 1 and a K-major A");
  LTM_REQUIRE(a.precision == 1 || a.precision == 3, "gemm: precision must be 1 (tf32) or 3 (split tf32)");
  const bool split = a.precision == 3;
  // 256-wide tiles (128 x 256 x 8 atoms) unless the problem is too small to give every SM a tile: then 128-wide
  // tiles double the CTA count and halve each tile's MMA time (one video: 12 -> 24 tiles)
  const long long tiles256 = (long long)((a.Nc + 255) / 256) * ((a.M + BM - 1) / BM) * a.batch;
  const int bn = (a.Nc > 128 && tiles256 >= 74) ? 256 : 128;
  const int K1 = two ? a.K1 : a.K;
  CUtensorMap mA, mB, mB2;
  if (a.a_group > 0) {
    // A rows in groups: dims {K, a_group, M / a_group}, box {32, min(a_group, 128), 128 / a_group (>= 1)}
    LTM_REQUIRE(a.a_kmajor && a.batch == 1, "gemm: grouped A rows need a K-major A and batch == 1");
    LTM_REQUIRE((BM % a.a_group == 0 || a.a_group % BM == 0) && a.M % a.a_group == 0,
                "gemm: a_group=%d must divide %d or be a multiple of it, and divide M=%d", a.a_group, BM, a.M);
    const int al = half ? 8 : 4;                       // pitch granularity in elements (16 bytes)
    LTM_REQUIRE(aligned16(a.A) && a.lda % al == 0 && a.lda >= a.K && a.a_group_stride % al == 0 &&
                a.a_group_stride >= (long long)a.a_group * a.lda, "gemm: grouped A pitches");
    const unsigned long long esz = half ? 2ull : 4ull;
    cuuint64_t dims[3] = {(cuuint64_t)a.K, (cuuint64_t)a.a_group, (cuuint64_t)(a.M / a.a_group)};
    cuuint64_t strides[2] = {(cuuint64_t)a.lda * esz, (cuuint64_t)a.a_group_stride * esz};
    cuuint32_t box[3] = {half ? 64u : 32u, (cuuint32_t)(a.a_group < BM ? a.a_group : BM),
                         (cuuint32_t)(a.a_group < BM ? BM / a.a_group : 1)};
    cuuint32_t estr[3] = {1u, 1u, 1u};
    CUresult r = g_encode(&mA, half ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3,
                          const_cast<float*>(a.A), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                          CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    LTM_REQUIRE(r == CUDA_SUCCESS, "gemm: cuTensorMapEncodeTiled(grouped A) failed with CUresult %d", (int)r);
  } else if (encode_operand(&mA, a.A, a.M, a.K, a.lda, a.strideA, a.batch, a.a_kmajor, BM, "A", half)) return -1;
  if (encode_operand(&mB, a.B, a.Nc, K1, a.ldb, a.strideB, a.batch, a.b_kmajor, bn, "B", half)) return -1;
  if (two) {
    if (encode_operand(&mB2, a.B2, a.Nc, a.K - K1, a.ldb2, a.strideB2, a.batch, a.b_kmajor, bn, "B2", half)) return -1;
  } else {
    mB2 = mB;
  }
  GemmDev d{};
  d.C = a.C; d.bias = a.bias; d.ldc = a.ldc; d.strideC = a.strideC;
  d.M = a.M; d.Nc = a.Nc; d.K = a.K; d.K1 = K1; d.batch = a.batch;
  d.a_kmajor = a.a_kmajor ? 1 : 0; d.b_kmajor = a.b_kmajor ? 1 : 0;
  d.CT = a.CT; d.ct_cols = a.ct_cols; d.ct_group = a.ct_group;
  d.c_group = a.c_group; d.c_group_stride = a.c_group_stride; d.bias_stride = a.bias_stride;
  d.mn_layout = MN_TF32.layout; d.mn_lbo = MN_TF32.lbo; d.mn_sbo = MN_TF32.sbo; d.mn_kadv = MN_TF32.kadv;
  if (half) {
    // 16-bit MN-major SWIZZLE_128B: atoms of [8 k][64 mn], MN atoms one 8 KB slab apart (LBO), 8-row k groups 1024 B
    // apart (SBO); one MMA (K = 16) advances two groups
    d.mn_layout = 2u; d.mn_lbo = 64u * 128u; d.mn_sbo = 1024u; d.mn_kadv = 2048u;
  }
  d.round_tf32 = a.round_tf32;
  d.ab_half = half;
  d.c_vec = (a.ldc % 4 == 0 && a.strideC % 4 == 0 && a.c_group_stride % 4 == 0 && aligned16(a.C) &&
             (a.CT == nullptr || a.ct_cols % 4 == 0)) ? 1 : 0;
  // fp16 output: a 16-byte store holds 8 halves, so every term of its address (row pitch, batch stride, group stride,
  // the base of C and of C_lo) must be a multiple of 8 halves; otherwise the epilogue stores halves one by one
  d.c_vec8 = (a.c_fp16 && a.ldc % 8 == 0 && a.strideC % 8 == 0 && a.c_group_stride % 8 == 0 && aligned16(a.C) &&
              (a.C_lo == nullptr || aligned16(a.C_lo))) ? 1 : 0;
  d.a_group = a.a_group;
  d.c_half = a.c_fp16 ? 1 : 0;
  d.C_lo = a.c_fp16 ? a.C_lo : nullptr;
  d.max_ctas = a.max_ctas;
  LTM_REQUIRE(a.C_lo == nullptr || (a.c_fp16 && aligned16(a.C_lo)), "gemm: C_lo needs c_fp16 and 16-byte alignment");
  LTM_REQUIRE(!a.c_fp16 || a.CT == nullptr, "gemm: fp16 output has no transposed store");
  d.a_batched = a.strideA != 0; d.b_batched = a.strideB != 0; d.b2_batched = a.strideB2 != 0; d.has_b2 = two ? 1 : 0;
  if (n_ext != nullptr || k_ext != nullptr) {      // ltm_gemm_extents: fp16 operands, precision 1, fp32 C (checked there)
    d.n_ext = n_ext; d.k_ext = k_ext;
    return bn == 256 ? launch_cfg<256, 4, false, false, true>(mA, mB, mB2, d, a.batch, stream)
                     : launch_cfg<128, 6, false, false, true>(mA, mB, mB2, d, a.batch, stream);
  }
  if (d.c_half) {           // fp16 output (the projected-memory K|V; Qt of the short-term attention)
    if (split) return bn == 256 ? launch_cfg<256, 2, true, true>(mA, mB, mB2, d, a.batch, stream)
                                : launch_cfg<128, 4, true, true>(mA, mB, mB2, d, a.batch, stream);
    return bn == 256 ? launch_cfg<256, 4, false, true>(mA, mB, mB2, d, a.batch, stream)
                     : launch_cfg<128, 6, false, true>(mA, mB, mB2, d, a.batch, stream);
  }
  if (split && bn == 256) return launch_cfg<256, 2, true>(mA, mB, mB2, d, a.batch, stream);
  if (split) return launch_cfg<128, 4, true>(mA, mB, mB2, d, a.batch, stream);
  if (bn == 256) return launch_cfg<256, 4, false>(mA, mB, mB2, d, a.batch, stream);
  return launch_cfg<128, 6, false>(mA, mB, mB2, d, a.batch, stream);
}

}  // namespace ltm

static int gemm_checked(const ltm_gemm_args* args, const int32_t* n_ext, const int32_t* k_ext, void* stream) {
  using namespace ltm;
  LTM_REQUIRE(args != nullptr, "gemm: null argument block");
  const ltm_gemm_args& a = *args;
  LTM_REQUIRE(a.A && a.B && a.C, "gemm: null operand");
  LTM_REQUIRE(ltm::aligned16(a.C) && a.strideC % 4 == 0, "gemm: C must be 16-byte aligned with a batch stride multiple of 4");
  LTM_REQUIRE(a.bias == nullptr || ltm::aligned16(a.bias), "gemm: bias must be 16-byte aligned");
  LTM_REQUIRE(a.M > 0 && a.Nc > 0 && a.K > 0 && a.batch > 0, "gemm: bad shape M=%d N=%d K=%d batch=%d", a.M, a.Nc,
              a.K, a.batch);
  LTM_REQUIRE(a.CT == nullptr || (a.ct_cols > 0 && a.ct_cols % 32 == 0 && a.ct_cols <= a.Nc && a.ct_group > 0 &&
                                  a.ct_group % 32 == 0 && a.M % a.ct_group == 0),
              "gemm: transposed store needs ct_cols %% 32 == 0, ct_group %% 32 == 0 and M %% ct_group == 0");
  LTM_REQUIRE(a.CT == nullptr || a.batch == 1, "gemm: transposed store is defined for batch == 1");
  LTM_REQUIRE(!(a.c_fp16 && a.impl == 1), "gemm: fp16 output exists in the tcgen05 kernel only");
  if (a.impl == 1) return gemm_simt_launch(a, (cudaStream_t)stream);
  LTM_REQUIRE(a.impl == 0, "gemm: unknown impl %d", a.impl);
  return gemm_tcgen05_launch(a, (cudaStream_t)stream, n_ext, k_ext);
}

extern "C" int ltm_gemm(const ltm_gemm_args* args, void* stream) { return gemm_checked(args, nullptr, nullptr, stream); }

extern "C" int ltm_gemm_extents(const ltm_gemm_args* args, const int32_t* n_ext, const int32_t* k_ext, void* stream) {
  using namespace ltm;
  LTM_REQUIRE(args != nullptr, "gemm_extents: null argument block");
  const ltm_gemm_args& a = *args;
  LTM_REQUIRE(a.ab_fp16 && a.precision == 1 && a.impl == 0,
              "gemm_extents: only fp16 operands with precision 1 on tcgen05 (ab_fp16=%d precision=%d impl=%d)", a.ab_fp16,
              a.precision, a.impl);
  LTM_REQUIRE((a.B2 == nullptr || a.K1 >= a.K) && a.CT == nullptr && !a.c_fp16 && a.a_group == 0,
              "gemm_extents: B2, the transposed store, fp16 output and grouped A rows are not supported");
  return gemm_checked(args, n_ext, k_ext, stream);
}

extern "C" int ltm_project_kv_t(const float* Bcoef, const float* Wkv, const float* bkv, float* Kt, float* V, int M,
                                int e, int D, int N, int precision, int impl, void* stream) {
  ltm_gemm_args a;
  memset(&a, 0, sizeof(a));
  a.A = Bcoef; a.lda = e; a.strideA = 0; a.a_kmajor = 1;
  a.B = Wkv; a.ldb = e; a.strideB = 0; a.b_kmajor = 1;
  a.B2 = nullptr; a.K1 = e;
  a.bias = bkv;
  a.C = V; a.ldc = D; a.strideC = 0;
  a.CT = Kt; a.ct_cols = D; a.ct_group = N;
  a.M = M; a.Nc = 2 * D; a.K = e; a.batch = 1;
  a.precision = precision; a.impl = impl;
  return ltm_gemm(&a, stream);
}

static int project_kv_impl(const float* Bcoef, const float* Wkv, const float* bkv, float* KV, int M, int e, int D2,
                           int precision, int impl, int round_tf32, void* stream) {
  ltm_gemm_args a;
  memset(&a, 0, sizeof(a));
  a.A = Bcoef; a.lda = e; a.strideA = 0; a.a_kmajor = 1;
  a.B = Wkv; a.ldb = e; a.strideB = 0; a.b_kmajor = 1;
  a.B2 = nullptr; a.K1 = e;
  a.bias = bkv;
  a.C = KV; a.ldc = D2; a.strideC = 0;
  a.M = M; a.Nc = D2; a.K = e; a.batch = 1;
  a.precision = precision; a.impl = impl; a.round_tf32 = round_tf32;
  return ltm_gemm(&a, stream);
}
extern "C" int ltm_project_kv(const float* Bcoef, const float* Wkv, const float* bkv, float* KV, int M, int e,
                              int D2, int precision, int impl, void* stream) {
  return project_kv_impl(Bcoef, Wkv, bkv, KV, M, e, D2, precision, impl, 0, stream);
}
extern "C" int ltm_project_kv_r(const float* Bcoef, const float* Wkv, const float* bkv, float* KV, int M, int e,
                                int D2, int precision, int impl, void* stream) {
  using namespace ltm;
  LTM_REQUIRE(impl == 0, "project_kv_r: the rounding epilogue exists in the tcgen05 kernel only");
  return project_kv_impl(Bcoef, Wkv, bkv, KV, M, e, D2, precision, impl, 1, stream);
}
