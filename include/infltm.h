/*
 * infltm.h -- C ABI of the B200-native infinity-Video LTM consolidation path (libinfltm.so).
 *
 * The reference (deep-spin/Infinite-Video) is pure Python; the interface this library sits under
 * is `LongTermAttention.forward(k, q, new_doc, layer_n)`
 * (infty-Video-LLaMA/InfVideoLLaMA/models/long_term_attention_gibbs.py:288-346, live "gibbs"
 * variant; .../long_term_attention.py:259-392, Gaussian variant).  The Python mirror of that class
 * (infinite_video_b200/ltm.py) binds these entry points with ctypes; see INTEGRATION.md.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer to caller-owned memory unless the name ends in `_host`;
 *     tensors are contiguous row-major; fp32 unless stated; indices int32; uniforms fp64.
 *   - `stream` is a cudaStream_t passed as void*; nothing here synchronises or allocates device
 *     memory (exception: the *_host entry points enqueue cudaMemcpyAsync on `stream`).
 *   - return 0 on success, <0 on error; ltm_last_error() gives the thread-local message.
 *   - symbols: Bv videos, L frames per chunk, T tokens per frame, e encoder width, N basis
 *     functions, S=512 re-samples, H heads, d head size, D=H*d, Q queries.
 */
#ifndef INFLTM_H
#define INFLTM_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LTM_STICKY_EDGES 129

int         ltm_version(void);
const char* ltm_last_error(void);
/* 0 when the loaded binary carries sm_100a code and a tcgen05-capable device is current */
int         ltm_device_check(void);

/* ---- R4: frame pooling.  gibbs:304  `k.reshape(B,L,T,e).mean(dim=2)`
 * k[Bv,L,T,e] -> xpart[Bv,L,splits,e]; the mean of frame l is sum_s xpart[.,l,s,:]. */
int ltm_pool_mean(const float* k, float* xpart, int Bv, int L, int T, int e, int splits, void* stream);
/* same with a bounded (persistent) grid of max_ctas CTAs (0 = one CTA per frame-split): used when the pooling
 * of the next chunk runs on a side stream under the compute-bound kernels of the current chunk. */
int ltm_pool_mean_grid(const float* k, float* xpart, int Bv, int L, int T, int e, int splits, int max_ctas,
                       void* stream);

/* frame pooling that also writes the chunk as IEEE fp16 (round to nearest even) to k16[Bv,L,T,e]: one pass over the
 * chunk serves the LTM and the kind::f16 short-term attention of the caller (SURVEY 8f N1) */
int ltm_pool_mean_convert(const float* k, float* xpart, void* k16, int Bv, int L, int T, int e, int splits,
                          void* stream);

/* Frame pooling folded with the first half of the regression of an UPDATE chunk: fbin_ptr[rows+1] lists, per basis
 * bin that receives new frames, its (consecutive) frames [fbin_ptr[r], fbin_ptr[r+1]); xbin[Bv,rows,e] receives the
 * sum of their pooled means (each frame pooled exactly like ltm_pool_mean with splits == 1).  The consolidation then
 * takes xbin as its frame operand (L = rows, splits = 1) with tables whose frame members are the bins
 * (ltm_rect_step_args.binned).  long_term_attention_gibbs.py:304 + :217-219. */
int ltm_pool_bins(const float* k, float* xbin, const int32_t* fbin_ptr, int Bv, int L, int T, int e, int rows,
                  void* stream);

/* same for a 16-bit chunk (fp16 when is_bf16 == 0, else bfloat16; the VideoChat2 Q-former runs under fp16
 * autocast): 128-bit loads of 8 elements, fp32 accumulation, fp32 output.  e % 8 == 0. */
int ltm_pool_mean_16(const void* k, int is_bf16, float* xpart, int Bv, int L, int T, int e, int splits,
                     void* stream);
/* same with a bounded (persistent) grid of max_ctas CTAs (0 = one CTA per frame-split, i.e. ltm_pool_mean_16): the
 * pooling of the next 16-bit chunk beside the current step.  Every frame-split is pooled by the same code for any
 * max_ctas, so xpart carries the same bits. */
int ltm_pool_mean_16_grid(const void* k, int is_bf16, float* xpart, int Bv, int L, int T, int e, int splits,
                          int max_ctas, void* stream);

/* ---- frame pooling of a ragged batch: k[Bv, L, T, e] is padded, video v uses its first lengths[v] frames
 * (0 = none), given as offs[Bv+1] = the exclusive prefix sum of the lengths (frames = offs[Bv]).
 * xpart[frames, splits, e] receives the pooled frames packed in video order, each bit-identical to ltm_pool_mean with
 * the same splits.  Only the frames listed are read.  max_ctas > 0 bounds the grid (persistent CTAs).
 * dtype: 0 fp32, 1 fp16, 2 bfloat16 (16-bit: e % 8 == 0, ltm_pool_mean_16's summation). */
int ltm_pool_mean_ragged(const void* k, int dtype, float* xpart, const int32_t* offs, int Bv, int L, int T, int e,
                         int splits, int frames, int max_ctas, void* stream);
/* ltm_pool_mean_ragged with each video's chunk at its own address: ptrs[Bv] (device) holds the base address of video
 * v's tokens, and frame l of video v is read at ptrs[v] + l*T*e elements, for l < offs[v+1] - offs[v].  The videos may
 * be separate tensors, views into one tensor holding a whole video, or views into one packed tensor; nothing is copied
 * into a padded chunk first.  xpart[frames, splits, e] is bit-identical to ltm_pool_mean_ragged over the same frames.
 * The caller guarantees what the library cannot check without reading the table: the pointer of every video with
 * frames is 16-byte aligned and its lengths[v]*T rows of e elements are dense (row pitch e).  The pointers of idle
 * videos are not read.  dtype, e, splits and max_ctas as ltm_pool_mean_ragged. */
int ltm_pool_mean_ptrs(const void* const* ptrs, int dtype, float* xpart, const int32_t* offs, int Bv, int L, int T,
                       int e, int splits, int frames, int max_ctas, void* stream);
/* ragged twin of ltm_pool_mean_convert (fp32 chunk k[Bv, L, T, e], lengths as offs[Bv+1] above): xpart as
 * ltm_pool_mean_ragged writes it for the same splits, and the chunk as IEEE fp16 padded per video,
 * k16[Bv, ld16, e] (ld16 % 64 == 0, ld16 >= L*T): with n_v = lengths[v]*T, tokens [0, n_v) of video v hold the
 * round-to-nearest-even cast, tokens [n_v, roundup64(n_v)) hold +0.0, and nothing past that is written -- the zero
 * tail lets the short-term GEMMs run whole 64-token k-blocks (ltm_gemm_extents).  Only the frames listed are read. */
int ltm_pool_mean_convert_ragged(const float* k, float* xpart, void* k16, const int32_t* offs, int Bv, int L, int T,
                                 int e, int splits, int frames, int ld16, void* stream);

/* ---- R6: sticky histogram of the previous call's density.  gibbs:196-203 (+score :224-230,
 * compute_probability :232-249).  scores[Bv,H,Q,N] -> hist_part[Bv,H,127] (sum over q; the sum
 * over heads happens in ltm_resample).  Normally fused into ltm_cont_attn_rect. */
int ltm_sticky_hist_rect(const float* scores, const int32_t* jb, const float* tb, float* hist_part,
                         int Bv, int H, int Q, int N, void* stream);

/* same, one partial histogram per (head, query tile of 32): hist_part[Bv, H*ceil(Q/32), 127] -- the layout the fused
 * attention kernels write */
int ltm_sticky_hist_rect_tiles(const float* scores, const int32_t* jb, const float* tb, float* hist_part,
                               int Bv, int H, int Q, int N, void* stream);

/* ---- R12 side output (Video-LLaMA copy only, gibbs:320-343 -> ./alphas_uniform -> relevant_frames.py):
 * scores[Bv,H,Q,N] -> out[Q,Bv,H,768]: Gibbs density on linspace(0,.25,256) | (.25,.5,256) | (.5,1,256), each segment
 * normalised by its trapezoid integral (weights wd[768]), the concatenation normalised to sum 1.  jd[768] = basis
 * index of each point (-1 none). */
int ltm_density_rect(const float* scores, const int32_t* jd, const float* wd, float* out,
                     int Bv, int H, int Q, int N, void* stream);

/* ---- G3: sticky histogram from the previous (mu, sigma).  long_term_attention.py:220-229.
 * mu,sd[Bv,R] -> hist_part[Bv,parts,128] (un-normalised): part p sums a contiguous share of the R rows;
 * ltm_resample adds the parts in a fixed order. */
int ltm_sticky_hist_gauss(const float* mu, const float* sd, const float* tb, float* hist_part,
                          int Bv, int R, int parts, void* stream);

/* ---- R7/G3: inverse-CDF re-sampling == Categorical(p).sample((S,)) with explicit uniforms.
 * gibbs:204-208, gauss:230-238.  hist_part[Bv,parts,ncat] is summed over `parts` in a fixed
 * order; normalize!=0 applies the reference's two p/sum(p) passes first.  CDF = sequential fp32
 * running sum / total, last entry forced to 1, draw -> first category with cdf >= u (fp64).
 * Outputs (any may be NULL): p_out[Bv,ncat] the probabilities used; b_draw[Bv,S] bins in draw
 * order; b_used[Bv,S] bins as consumed (sorted ascending when sort!=0, the Gaussian variant);
 * ts[Bv,S]=bins[b_used]; idx[Bv,S]=bin2basis[b_used] (bin2basis may be NULL -> idx=b_used). */
int ltm_resample(const float* hist_part, int parts, int ncat, int normalize, const double* u,
                 const float* bins, const int32_t* bin2basis, int sort,
                 float* p_out, int32_t* b_draw, int32_t* b_used, float* ts, int32_t* idx,
                 int Bv, int S, void* stream);

/* ---- R3/R5/R8: memory contraction + regression for rectangular bases.  gibbs:184-222.
 * The ridge operator has <=1 non-zero per row, so B = G^T [xm ; x] is a segmented mean:
 *   B_new[v,j,:] = g[j] * sum_{p in seg(j)} row(p),  row(p) = B_past[v, idx[v,p], :] for p < S
 *   (zero row when idx < 0), else the pooled frame p-S.  Table set 0 (first chunk, members are
 *   frame indices) is used where new_doc[v] != 0 (or B_past == NULL), table set 1 otherwise. */
int ltm_consolidate_rect(const float* B_past, const float* xpart, const int32_t* idx,
                         const uint8_t* new_doc,
                         const int32_t* seg_ptr0, const int32_t* seg_mem0, const float* g0,
                         const int32_t* seg_ptr1, const int32_t* seg_mem1, const float* g1,
                         float* B_new, int Bv, int N, int e, int L, int splits, int S, void* stream);
/* same, additionally writing B_new as IEEE fp16 to B_half[Bv,N,e] (round to nearest; NULL = off): the operand of
 * the fp16 K/V projection (ltm_gemm ab_fp16) */
int ltm_consolidate_rect_h(const float* B_past, const float* xpart, const int32_t* idx,
                           const uint8_t* new_doc,
                           const int32_t* seg_ptr0, const int32_t* seg_mem0, const float* g0,
                           const int32_t* seg_ptr1, const int32_t* seg_mem1, const float* g1,
                           float* B_new, void* B_half, int Bv, int N, int e, int L, int splits, int S, void* stream);

/* ---- projected-memory state (the K/V projection is affine and the memory contraction is linear): the keys / values
 * of the bins that hold only re-sampled memory follow from the previous call's keys / values,
 *   KV_new[v,j,:] = g[j] * sum_{p in seg(j), idx[v,p] >= 0} KV_past[v, idx[v,p], :] + (1 - g[j] * cnt) * bkv      j < jf
 * (cnt = number of members with a valid index), so that only the rows j >= jf that receive new frames go through the
 * projection GEMM (a quarter of them at tau = 0.75).  Same launch as ltm_consolidate_rect_h: B_new is produced as
 * before; the KV rows j < jf are written only for videos that take the update branch.  round_tf32 == 1 stores the KV
 * rows rounded to the tf32 grid (operands of the tensor-core attention); round_tf32 == 2: KV_past / KV_new point to
 * IEEE fp16 storage [Bv, N, ldkv] (fp32 accumulation, one rounding at the store; ldkv % 8 == 0).  idx_stride: elements between the index
 * rows of consecutive videos (S; 0 = one row shared by all videos, the uniform re-sampling table).
 * KV_past / KV_new: [Bv, N, ldkv] with ldkv = 2D; KV_past == NULL: coefficients only. */
int ltm_consolidate_rect_kv(const float* B_past, const float* xpart, const int32_t* idx, int64_t idx_stride,
                            const uint8_t* new_doc,
                            const int32_t* seg_ptr0, const int32_t* seg_mem0, const float* g0,
                            const int32_t* seg_ptr1, const int32_t* seg_mem1, const float* g1,
                            float* B_new, void* B_half,
                            const float* KV_past, float* KV_new, const float* bkv, int ldkv, int jf, int round_tf32,
                            int Bv, int N, int e, int L, int splits, int S, void* stream);

/* ---- batched GEMM on tcgen05 tensor cores (kind::tf32, fp32 operands fed by TMA, fp32
 * accumulate in TMEM).  C[b] (M x Nc, ldc) = A[b] (M x K) * B[b] (K x Nc) (+ bias[Nc]).
 *   a_kmajor: A[b] stored [M][K] (K contiguous, lda = row pitch) else [K][M] (lda = pitch of a K row)
 *   b_kmajor: B[b] stored [Nc][K] (K contiguous)              else [K][Nc]
 *   B may be split along K: rows [0,K1) come from B, rows [K1,K) from B2 (same layout rules);
 *   pass B2 = NULL, K1 = K for a single segment.
 *   batch strides in elements (0 = operand shared by all batches).
 *   precision: 1 = single-pass TF32; 3 = split hi/lo 3-pass (fp32-grade accuracy).
 *   impl: 0 = tcgen05 (product path), 1 = fp32 SIMT check kernel (tests/debug only). */
typedef struct {
  const float* A;  int64_t lda;  int64_t strideA;  int a_kmajor;
  const float* B;  int64_t ldb;  int64_t strideB;  int b_kmajor;
  const float* B2; int64_t ldb2; int64_t strideB2; int K1;
  const float* bias;
  float* C;        int64_t ldc;  int64_t strideC;
  int M, Nc, K, batch;
  int precision;
  int impl;
  /* optional transposed store: columns [0, ct_cols) of the product go to CT instead of C, transposed inside
   * groups of ct_group consecutive rows: CT[(m / ct_group) * ct_cols + c][m % ct_group]; the remaining columns
   * c >= ct_cols go to C[m * ldc + (c - ct_cols)].  ct_cols % 32 == 0, ct_group % 32 == 0.  CT = NULL: off. */
  float* CT; int ct_cols; int ct_group;
  /* optional two-level row mapping of C: row m lives at (m / c_group) * c_group_stride + (m % c_group) * ldc
   * (c_group = 0: plain m * ldc).  Lets a batched product land directly in [head][video][query] style layouts. */
  int c_group; int64_t c_group_stride;
  /* bias of batch b starts at bias + b * bias_stride */
  int64_t bias_stride;
  /* != 0: round the stored row-major results to the tf32 grid (round to nearest), for products that feed another
   * tf32 tensor-core contraction (the tensor core itself would truncate, which biases sums of products) */
  int round_tf32;
  /* != 0: A, B (and B2) point to IEEE fp16 data (leading dimensions / strides in elements, multiples of 8), both
   * A K-major, B K-major or MN-major; the products run as kind::f16 UMMAs with fp32 accumulation -- the same 11-bit
   * significand as tf32 at half the operand bytes and twice the MMA rate, for operands whose range fits fp16
   * (precision must be 1) */
  int ab_fp16;
  /* optional two-level row mapping of A (K-major A, batch == 1): row m lives at
   * A + (m / a_group) * a_group_stride + (m % a_group) * lda  -- e.g. the rows [jf, N) of every video's coefficient
   * matrix as one flat problem (A = B_new + jf * e, a_group = N - jf, a_group_stride = N * e).  a_group must divide
   * 128 or be a multiple of 128, and M % a_group == 0 (one TMA box spans 128 / a_group groups).  0 = plain m * lda. */
  int a_group; int64_t a_group_stride;
  /* != 0: C points to IEEE fp16 storage (ldc / strideC / c_group_stride in elements; round to nearest even): the
   * product feeds a kind::f16 tensor-core contraction whose operands carry the same 11-bit significand as tf32 */
  int c_fp16;
  /* with c_fp16: optional second fp16 output of the same layout, C_lo = rn(x - float(rn(x))) -- the result as two fp16
   * terms (22 significant bits), the operand format of the fp16x2 contractions (ltm_cont_attn_gauss_tc16).  NULL: off */
  void* C_lo;
  /* bound of the persistent grid (0 = one CTA per SM).  A contraction that runs BESIDE an HBM-bound kernel of another
   * stream (the K/V projection beside the next chunk's frame pooling) is not on the critical path, and confined to
   * fewer SMs it takes less of the L2 -> SM bandwidth the streaming kernel lives on at any one time: measured at the
   * NExT-QA shape, 148 -> 64 CTAs: the overlapped step 194.6 k -> 207.3 k chunks/s (the projection itself 0.09 -> 0.11 ms) */
  int max_ctas;
} ltm_gemm_args;
int ltm_gemm(const ltm_gemm_args* args, void* stream);
/* ltm_gemm with per-batch extents (device int32 arrays of `batch` entries, each optional = NULL): the tiles of batch b
 * whose first column is >= n_ext[b] are skipped (a tile that straddles n_ext[b] is computed and stored in full, up to
 * Nc), and batch b accumulates over its first k_ext[b] K-elements only (a multiple of 64, the fp16 k-block; the
 * operands must hold zeros in [K_b, roundup64) if K_b itself is not).  A batch with either extent 0 gets no tiles: its
 * C is not written.  Supported: ab_fp16 with precision 1 and fp32 C (no B2, CT, c_fp16 or a_group). */
int ltm_gemm_extents(const ltm_gemm_args* args, const int32_t* n_ext, const int32_t* k_ext, void* stream);

/* ---- R9: K/V projection.  gibbs:312-313  keys=proj_key(B), values=proj_value(B).
 * KV[M, 2D] = Bcoef[M, e] * Wkv[2D, e]^T + bkv   (M = Bv*N; Wkv = [W_key ; W_value]). */
int ltm_project_kv(const float* Bcoef, const float* Wkv, const float* bkv, float* KV,
                   int M, int e, int D2, int precision, int impl, void* stream);

/* same projection, keys stored transposed per head for the fast attention path:
 * Kt[Bv, H, 64, N] (= [M/N][D][N]) and V[M, D]. */
int ltm_project_kv_t(const float* Bcoef, const float* Wkv, const float* bkv, float* Kt, float* V,
                     int M, int e, int D, int N, int precision, int impl, void* stream);

/* ---- R10/R11 (+R6 fused): continuous attention over rectangular bases.  gibbs:224-286,:346.
 * r_j = W_j e^{S_j} / (sum_i W_i e^{S_i} + W_out),  S = (q_h/sqrt(d)) K_h^T,  ctx = r V.
 * q[Bv,Q,D], KV[Bv,N,2D] -> ctx[Bv,Q,D]; optional scores_out[Bv,H,Q,N];
 * optional hist_part[Bv, H*ceil(Q/32), 127] (next call's sticky histogram partials). */
int ltm_cont_attn_rect(const float* q, const float* KV, const float* W, float W_out,
                       const int32_t* jb, const float* tb,
                       float* ctx, float* scores_out, float* hist_part,
                       int Bv, int Q, int N, int H, int d, void* stream);

/* ---- G4: continuous attention, Gaussian closed form.  long_term_attention.py:286-325.
 * a = softmax(20 S); mu = a.mu_b; var = a.(mu_b^2+sigma_b^2) - mu^2;
 * r_j = N(mu; mu_j, sigma_j^2 + var); ctx = r V.  Also writes mu_out, sd_out [Bv, H*Q]. */
int ltm_cont_attn_gauss(const float* q, const float* KV, const float* basis_mu, const float* basis_sigma,
                        float* ctx, float* scores_out, float* mu_out, float* sd_out,
                        int Bv, int Q, int N, int H, int d, void* stream);

/* ---- G4 optional output: KL(N(mu, sd^2) || N(mu_0, sigma_0^2)) per row, long_term_attention.py:296-304 (including
 * its quirk: the mean term is dropped when mu_0 > 0).  mu, sd, out: [n]. */
int ltm_kl_gauss(const float* mu, const float* sd, float mu_0, float sigma_0, float* out, int64_t n, void* stream);

/* ---- fast path of both attention variants for num_basis in {64,128,256}, head_size 64: keys transposed
 * (Kt[Bv,H,64,N], from ltm_project_kv_t), values V[Bv,N,ldv].  Same outputs as the two functions above. */
int ltm_attn_fast_supported(int N, int d);
int ltm_cont_attn_rect_t(const float* q, const float* Kt, const float* V, int64_t ldv, const float* W, float W_out,
                         const int32_t* jb, const float* tb, float* ctx, float* scores_out, float* hist_part,
                         int Bv, int Q, int N, int H, int d, void* stream);
int ltm_cont_attn_gauss_t(const float* q, const float* Kt, const float* V, int64_t ldv, const float* basis_mu,
                          const float* basis_sigma, float* ctx, float* scores_out, float* mu_out, float* sd_out,
                          int Bv, int Q, int N, int H, int d, void* stream);

/* ---- tensor-core path of the rect attention for num_basis in {64,128,256}, head_size 64 (csrc/attn_tc.cu): both
 * contractions as tf32 UMMAs.  K[Bv*N, ldkv], V[Bv*N, ldkv] row-major (head h at column h*64; e.g. the two halves
 * of ltm_project_kv's KV, ldkv = 2D), already rounded to tf32 (ltm_gemm round_tf32 / ltm_project_kv_r).
 * X[N,32]: extra operand rows (1, hi/lo of c_j/W_j; infinite_video_b200/tables.py), c_none: trapezoid node weight
 * of the sticky edges outside every basis.  Outputs as ltm_cont_attn_rect. */
int ltm_attn_tc_supported(int N, int d);
int ltm_cont_attn_rect_tc(const float* q, const float* K, const float* V, int64_t ldkv, const float* X,
                          const float* W, float W_out, float c_none, const int32_t* jb, const float* tb,
                          float* ctx, float* scores_out, float* hist_part,
                          int Bv, int Q, int N, int H, int d, void* stream);
/* num_basis 512 on the same kernel: every (query tile, head, video) is split into two work items over the halves of
 * the basis range, merged by a small combine kernel (online-softmax rescaling); the next call's sticky histogram is
 * computed from the stored scores.  scores_ws[Bv,H,Q,N] and part_ws[ltm_attn_tc_split_workspace_floats(Bv,Q,H)] are
 * caller-provided workspaces (scores_ws doubles as the optional scores output). */
int ltm_attn_tc_split_supported(int N, int d);
int64_t ltm_attn_tc_split_workspace_floats(int Bv, int Q, int H);
int ltm_cont_attn_rect_tc_split(const float* q, const float* K, const float* V, int64_t ldkv, const float* X,
                                const float* W, float W_out, const int32_t* jb, const float* tb,
                                float* ctx, float* scores_ws, float* part_ws, float* hist_part,
                                int Bv, int Q, int N, int H, int d, void* stream);
/* the same two entry points for K|V stored as IEEE fp16 (csrc/attn_tc.cu, KvF16: kind::f16 UMMAs, the same 11-bit
 * significand as the tf32 grid at half the bytes).  K, V: fp16 [Bv*N, ldkv] (ldkv in halves, % 8 == 0; e.g. the two
 * halves of an fp16 KV[Bv,N,2D] from ltm_gemm c_fp16 / ltm_consolidate_rect_kv round_tf32 == 2); X16: fp16 [N,64]
 * (columns 0..2 = 1, hi, lo of c_j / W_j; infinite_video_b200/tables.py).  q, W, outputs as above (fp32). */
int ltm_cont_attn_rect_tc16(const float* q, const void* K, const void* V, int64_t ldkv, const void* X16,
                            const float* W, float W_out, float c_none, const int32_t* jb, const float* tb,
                            float* ctx, float* scores_out, float* hist_part,
                            int Bv, int Q, int N, int H, int d, void* stream);
int ltm_cont_attn_rect_tc16_split(const float* q, const void* K, const void* V, int64_t ldkv, const void* X16,
                                  const float* W, float W_out, const int32_t* jb, const float* tb,
                                  float* ctx, float* scores_ws, float* part_ws, float* hist_part,
                                  int Bv, int Q, int N, int H, int d, void* stream);
/* ltm_project_kv with the stored K and V rounded to tf32 */
int ltm_project_kv_r(const float* Bcoef, const float* Wkv, const float* bkv, float* KV,
                     int M, int e, int D2, int precision, int impl, void* stream);

/* ---- G1: Gaussian RBF evaluation.  basis_functions.py:158-164.
 * out[p, j] (ld) = N(t_p; mu_j, sigma_j^2); t may be gathered: t_p = tvals[tidx[p]] when tidx != NULL. */
int ltm_rbf_eval(const float* tvals, const int32_t* tidx, const float* basis_mu, const float* basis_sigma,
                 float* out, int64_t ld, int P, int N, void* stream);

/* ---- G2: ridge operator  G = F^T (F F^T + ridge I)^-1 for the Gaussian design matrix, solved in
 * fp64 on the device.  long_term_attention.py:70-86.  positions[P] (padded), rows [trim, trim+rows)
 * are kept.  Outputs (either may be NULL): G[rows, N] and GT[N, rows] (row pitch ldgt >= rows) in fp32.
 * workspace: fp64, ltm_ridge_workspace_doubles(P, N) elements. */
int64_t ltm_ridge_workspace_doubles(int P, int N);
int ltm_ridge_solve(const float* positions, int P, int trim, int rows,
                    const float* basis_mu, const float* basis_sigma, int N, double ridge,
                    float* G, float* GT, int64_t ldgt, double* workspace, void* stream);

/* ---- gather rows: out[v, s, :] = src[v, idx[v,s], :]  (zero row when idx < 0) */
int ltm_gather_rows(const float* src, const int32_t* idx, float* out, int Bv, int rows_src, int S, int e,
                    void* stream);

/* ---- G4 on the tensor cores: continuous attention of the Gaussian variant (long_term_attention.py:286-325) with both
 * contractions as kind::f16 UMMAs over two-term operands (x ~ hi + lo: fp32-grade products).  KV_hi / KV_lo: fp16
 * [Bv*N, ldkv] from ltm_gemm (c_fp16 + C_lo), keys of head h at columns [h*d, (h+1)*d), values at H*d + the same.
 * Outputs ctx[Bv,Q,H*d], mu / sd [Bv, H*Q] (either may be NULL).  num_basis 64 / 128 / 256, head size 64. */
int ltm_cont_attn_gauss_tc16(const float* q, const void* KV_hi, const void* KV_lo, int64_t ldkv, const float* basis_mu,
                             const float* basis_sigma, float* ctx, float* mu_out, float* sd_out, int Bv, int Q, int N,
                             int H, int d, void* stream);

/* ---- variant G, sticky update without materialising the re-sampled rows: b_sorted[Bv,S] are the drawn bins in
 * ascending order (ltm_resample sort = 1), GT[N, >= S+L] the update operator G_inf^T (row pitch ldg).
 * out[v, n, b] = sum of GT[n, s] over the draws s with b_sorted[v,s] == b (b < nbins), out[v, n, nbins + l] = GT[n, S+l]:
 * out[v] [R ; k] == GT [xm ; k] with xm[s] = R[b_s].  long_term_attention.py:239-250. */
int ltm_fold_sample_columns(const float* GT, int64_t ldg, const int32_t* b_sorted, float* out, int Bv, int N, int S,
                            int L, int nbins, void* stream);

/* ---- whole per-chunk step of variant R for Bv videos (device buffers), and the same through
 * host buffers (H2D of k,q,u,new_doc and D2H of ctx enqueued on `stream`; caller synchronises).
 * ltm_rect_step with k == NULL skips the frame pooling and consumes a->xpart as already filled by an
 * earlier ltm_pool_mean (pooling does not depend on the memory state, so a host may issue it for the
 * next chunk on a second stream while this chunk's regression / projection / attention run). */
typedef struct {
  int Bv, L, T, e, N, Q, H, d, S, splits, sticky, precision, gemm_impl;
  /* constant tables (device) */
  const int32_t *seg_ptr0, *seg_mem0; const float* g0;
  const int32_t *seg_ptr1, *seg_mem1; const float* g1;
  const int32_t* jb; const float* tb; const float* bins; const int32_t* bin2basis;
  const int32_t* idx_uniform;           /* [S] used when sticky == 0 */
  const float* W; float W_out;
  const float *Wkv, *bkv;               /* [2D,e], [2D] */
  /* per-video state (device) */
  const float* B_past; float* B_new;    /* [Bv,N,e] ping-pong, caller swaps after the call */
  float* hist_part;                     /* [Bv, H*ceil(Q/32), 127] previous call's partials (in) and new (out) */
  /* workspace (device) */
  float* xpart;                         /* [Bv,L,splits,e] */
  float* KV;                            /* [Bv,N,2D] (generic attention path) */
  float* Kt; float* V;                  /* [Bv,H,64,N], [Bv,N,D]: fast path when N in {64,128,256} (else NULL) */
  int32_t *b_draw, *idx; float* ts;     /* [Bv,S] */
  float* p;                             /* [Bv,127] */
  float* scores;                        /* optional [Bv,H,Q,N] */
  /* device staging for the *_host entry point */
  void* k_dev; float* q_dev; double* u_dev; uint8_t* new_doc_dev; float* ctx_dev;
  /* optional cudaEvent_t pairs recorded on `stream` around each stage (NULL = skip):
   * [0,1] pool  [2,3] re-sample  [4,5] consolidate  [6,7] K/V projection  [8,9] attention */
  void* prof_events[10];
  /* tensor-core attention (used when X != NULL, KV != NULL, precision == 1 and ltm_attn_tc_supported(N, d)) */
  const float* X; float c_none;
  /* fp16 operands of the K/V projection (used with the tensor-core attention when both are set): B_half[Bv,N,e]
   * workspace (written by the consolidation), Wkv_half[2D,e] = Wkv in fp16.  Coefficients beyond the fp16 range
   * (|B| > 65504) become inf and propagate visibly; leave NULL for fp32 (tf32) operands. */
  void* B_half; const void* Wkv_half;
  /* projected-memory state (ltm_consolidate_rect_kv): KV_past[Bv,N,2D] = the previous call's K|V (ping-pong with KV,
   * caller swaps after the call), jf = first bin that holds a new frame in the update tables.  Used when KV_past != NULL,
   * jf > 0, every video takes the update branch (B_past != NULL, new_doc == NULL) and N - jf tiles 128 rows evenly;
   * otherwise all N rows are projected.  proj_precision: precision of the K/V projection GEMM (0 = `precision`). */
  const float* KV_past; int jf; int proj_precision;
  /* workspace of the two-half tensor-core attention (num_basis 512): ltm_attn_tc_split_workspace_floats(Bv,Q,H)
   * floats; with it (and `scores`) set, num_basis 512 takes ltm_cont_attn_rect_tc_split */
  float* attn_part;
  /* kv_half != 0: KV / KV_past point to IEEE fp16 storage [Bv,N,2D] and X16 (fp16 [N,64]) is set: the projection
   * GEMM stores fp16, the carried rows are accumulated in fp32 and stored as fp16, the attention runs on
   * ltm_cont_attn_rect_tc16.  Same significand as the tf32 grid of the fp32 layout; magnitudes beyond 65504 become inf. */
  int kv_half; const void* X16;
  /* binned != 0 (update calls of all videos only: B_past set, new_doc NULL): `xpart` holds / receives the bin sums of
   * ltm_pool_bins ([Bv, xb_rows, e]) instead of the pooled frames; fbin_ptr[xb_rows+1] is its frame table and
   * seg_ptr1b / seg_mem1b the update tables with the frames of a bin collapsed into one member S + r. */
  int binned, xb_rows;
  const int32_t* fbin_ptr; const int32_t* seg_ptr1b; const int32_t* seg_mem1b;
  /* grid bound of the K/V projection GEMM (ltm_gemm_args.max_ctas; 0 = one CTA per SM): set when the next chunk's
   * pooling runs beside this step */
  int gemm_ctas;
  /* ragged batch (lengths != NULL): video v uses the first lengths[v] frames of its padded chunk k[v, L*T, e]
   * (lengths[v] == 0: the video is idle this call).  frame_offs[Bv+1] is the exclusive prefix sum of lengths and
   * `frames` its total; `xpart` holds the pooled frames packed in that order, [frames, splits, e].  The tables of a
   * video are selected from the bank by its length: bank_seg_ptr0/1 [L+1, N+1] (absolute offsets into the
   * concatenated bank_seg_mem0/1), bank_g0/1 [L+1, N] (infinite_video_b200/tables.py RectBank).  `jf` must be the
   * smallest jf among the lengths of the videos that update.  new_doc flags apply to the videos that are present.
   * An idle video keeps its state bit for bit: its coefficient rows (zeros when B_past == NULL), K|V rows (when
   * KV_past is set; otherwise they are projected from the kept coefficients) and sticky histogram partials (saved in
   * hist_keep[Bv, H*ceil(Q/32), 127] during the call) carry over, its re-sampling is skipped (its row of u is not
   * read), and its ctx rows are zero.  n_idle: number of idle videos.  u may be NULL
   * when no video continues its memory.  Frame pooling per
   * bin (binned) does not apply.  lengths == NULL: lock-step, every field below is ignored. */
  const int32_t* lengths; const int32_t* frame_offs; int frames; int n_idle;
  const int32_t *bank_seg_ptr0, *bank_seg_mem0; const float* bank_g0;
  const int32_t *bank_seg_ptr1, *bank_seg_mem1; const float* bank_g1;
  float* hist_keep;
  /* storage of the chunk: k of ltm_rect_step, k_host and k_dev of ltm_rect_step_host.  0 fp32, 1 fp16, 2 bfloat16.
   * A 16-bit chunk (e % 8 == 0) is pooled per frame from its own storage with fp32 accumulation, in the summation
   * order of ltm_pool_mean_16 (lock-step) or ltm_pool_mean_ragged (ragged); it is never pooled per bin (binned == 0). */
  int k_dtype;
  /* chunk given per video (NULL = off): k_ptrs[Bv] (device) holds the base address of video v's tokens, pooled as
   * ltm_pool_mean_ptrs pools them; the ragged fields above must be set (lengths, frame_offs, frames) and k must be
   * NULL.  Not with binned.  The step pools the chunk from the table whenever it is set (ltm_rect_step_overlap: on the
   * compute stream, before the rest of the step). */
  const void* const* k_ptrs;
} ltm_rect_step_args;
int ltm_rect_step(const ltm_rect_step_args* a, const void* k, const float* q, const double* u,
                  const uint8_t* new_doc, float* ctx, void* stream);
int ltm_rect_step_host(const ltm_rect_step_args* a, const void* k_host, const float* q_host,
                       const double* u_host, const uint8_t* new_doc_host, float* ctx_host, void* stream);

/* ---- the same step with the frame pooling of the NEXT chunk issued beside it (two-stream schedule in one call):
 *   side:     wait(main) -> pool(k_next -> xpart_next) -> record ev_pooled_next
 *   compute:  wait(main), wait(ev_pooled_cur) -> re-sample / consolidate / project / attention of this chunk
 *             (a->xpart holds this chunk's pooled frames, filled by the previous call's side-stream pooling)
 *   main:     wait(compute)
 * Frame pooling does not depend on the memory state and is the HBM-bound 93 % of a call's bytes; the other kernels
 * are tensor- / latency-bound.  Streams and (timing-disabled) events are the caller's; the events are re-recorded
 * on every call.  k_next == next_ptrs == NULL issues no pooling; ev_pooled_cur == NULL waits for nothing.  The pooling of the
 * next chunk is bracketed by a->prof_events[0,1] when those are set. */
typedef struct {
  void *main_stream, *side_stream, *compute_stream;
  void *ev_fork_pool, *ev_pooled_cur, *ev_pooled_next, *ev_fork, *ev_join;
  const void* k_next; float* xpart_next; int pool_ctas;
  int next_binned;     /* pool k_next with ltm_pool_bins (the call that consumes it must set args.binned) */
  /* ragged next chunk (next_lengths != NULL): pool the first next_lengths[v] frames of each video of k_next (padded
   * to args.L frames) into xpart_next packed as [next_frames, next_splits, e] (ltm_pool_mean_ragged) */
  const int32_t* next_lengths; const int32_t* next_offs; int next_frames; int next_splits;
  int next_dtype;      /* storage of k_next, as ltm_rect_step_args.k_dtype (16-bit: next_binned == 0) */
  /* next chunk given per video, as ltm_rect_step_args.k_ptrs (NULL = off): needs next_lengths / next_offs, k_next must
   * be NULL and next_binned 0 */
  const void* const* next_ptrs;
} ltm_overlap;
int ltm_rect_step_overlap(const ltm_rect_step_args* a, const ltm_overlap* o, const float* q, const double* u,
                          const uint8_t* new_doc, float* ctx);

/* ---- N1 (caller, Qformer.py:279-304): row softmax of the short-term attention scores, in place.
 * S[rows, n] <- softmax(S * scale + mask[row / rows_per_mask, :]) (mask may be NULL); and the alpha blend
 * out = alpha * a + (1 - alpha) * b over n elements. */
int ltm_softmax_rows(float* S, const float* mask, int rows, int n, int rows_per_mask, float scale, void* stream);
int ltm_blend(const float* a, const float* b, float alpha, float* out, int64_t n, void* stream);
/* the same softmax with the probabilities written as IEEE fp16 to P16[rows, n] (S is scratch afterwards; rows of
 * n <= 8192 are held in registers: one pass over HBM, S untouched), and the
 * fp32 -> fp16 conversion (round to nearest even) of the chunk tokens: operands of the kind::f16 short-term GEMMs */
int ltm_softmax_rows_h(float* S, const float* mask, void* P16, int rows, int n, int rows_per_mask, float scale,
                       void* stream);
/* the fp16 softmax of a ragged batch: S[rows, ld] and P16[rows, ld] (ld % 64 == 0); row r belongs to video
 * v = r / rows_per_len and spans its first n_v = n_len[v] columns (n_len: device int32, rows / rows_per_len entries,
 * n_v <= ld), softmax(S * scale + mask[v, :n_v]) with mask rows of pitch mask_ld (may be NULL).  A row of n_v
 * columns is reduced in the order ltm_softmax_rows_h reduces a row of n = n_v.  P columns [n_v, roundup64(n_v)) are
 * written as 0, nothing beyond; columns >= n_v of S and of the mask are not read; rows with n_v = 0 are not touched. */
int ltm_softmax_rows_h_len(const float* S, const float* mask, void* P16, const int32_t* n_len, int rows, int ld,
                           int mask_ld, int rows_per_len, float scale, void* stream);
int ltm_to_half(const float* src, void* dst, int64_t n, void* stream);
/* fp32 [rows, K] -> fp16 [rows, 3K], x ~ hi + lo in three K segments per row: side 0 (A operand) [hi | lo | hi], side 1
 * (B operand) [hi | hi | lo].  A plain fp16 ltm_gemm (ab_fp16) over K' = 3K then computes a_hi b_hi + a_lo b_hi +
 * a_hi b_lo: the three-term product of the split-TF32 mode at the fp16 tensor rate. */
int ltm_split_half3(const float* src, void* dst, int64_t rows, int K, int side, void* stream);

/* ---- CUDA-event helpers so a ctypes host can time stages on the launching stream */
int ltm_event_create(void** ev);
int ltm_event_create_sync(void** ev);                             /* no timing: stream fork / join only */
int ltm_event_record(void* ev, void* stream);
int ltm_stream_wait_event(void* stream, void* ev);
int ltm_event_elapsed_ms(void* start, void* stop, float* ms);   /* synchronises on `stop` */
int ltm_event_destroy(void* ev);

#ifdef __cplusplus
}
#endif
#endif /* INFLTM_H */
