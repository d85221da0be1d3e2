// C-ABI glue: error reporting, device check, and the fused per-chunk step of variant R.
#include <stdarg.h>

#include "common.cuh"

namespace ltm {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

__global__ void arch_probe_kernel(int* out) {
#if defined(__CUDA_ARCH_FEAT_SM100_ALL) || defined(__CUDA_ARCH_SPECIFIC__) || (__CUDA_ARCH__ >= 1000)
  *out = __CUDA_ARCH__;
#else
  *out = -1;
#endif
}

}  // namespace ltm

extern "C" int ltm_version(void) { return 100; }   // 0.1.0

extern "C" const char* ltm_last_error(void) { return ltm::g_err; }

extern "C" int ltm_device_check(void) {
  using namespace ltm;
  int dev = 0;
  LTM_CUDA(cudaGetDevice(&dev));
  cudaDeviceProp prop;
  LTM_CUDA(cudaGetDeviceProperties(&prop, dev));
  LTM_REQUIRE(prop.major == 10, "device %s is sm_%d%d; libinfltm carries sm_100a code only", prop.name, prop.major,
              prop.minor);
  cudaFuncAttributes fa;
  LTM_CUDA(cudaFuncGetAttributes(&fa, arch_probe_kernel));
  return 0;
}

// Storage of a chunk (ltm_rect_step_args.k_dtype, ltm_overlap.next_dtype): 0 fp32, 1 fp16, 2 bfloat16.  A 16-bit chunk
// is read as 128-bit vectors of 8 elements and is never pooled per bin.
static int check_chunk_dtype(const char* who, const char* field, int dtype, int e, bool binned) {
  LTM_REQUIRE(dtype >= 0 && dtype <= 2, "%s: %s=%d (0 fp32, 1 fp16, 2 bfloat16)", who, field, dtype);
  LTM_REQUIRE(dtype == 0 || e % 8 == 0, "%s: a 16-bit chunk needs e %% 8 == 0 (e=%d)", who, e);
  LTM_REQUIRE(dtype == 0 || !binned, "%s: a 16-bit chunk is not pooled per bin", who);
  return 0;
}

// A chunk given per video (table: ltm_rect_step_args.k_ptrs, ltm_overlap.next_ptrs) is ragged, comes without a chunk
// pointer and is never pooled per bin.
static int check_chunk_table(const char* who, const char* field, const void* table, const void* k,
                             const int32_t* lengths, bool binned) {
  if (!table) return 0;
  LTM_REQUIRE(!k, "%s: %s and a chunk pointer are both set", who, field);
  LTM_REQUIRE(lengths, "%s: %s needs per-video lengths", who, field);
  LTM_REQUIRE(!binned, "%s: a chunk given per video (%s) is not pooled per bin", who, field);
  return 0;
}

// Frame pooling of one chunk of the geometry of `a` into xpart: packed frames of a ragged chunk (offs != NULL: frame
// offsets, `frames` in all; from the per-video table ptrs when set), per-bin sums (binned, fp32 chunks) or per-frame
// means.  dtype: storage of k, as checked by check_chunk_dtype.  max_ctas bounds the grid (0 = one CTA per unit).
static int pool_chunk(const ltm_rect_step_args* a, const void* k, const void* const* ptrs, int dtype, float* xpart,
                      const int32_t* offs, int frames, int splits, bool binned, int max_ctas, void* stream) {
  LTM_REQUIRE(!binned || a->fbin_ptr, "frame pooling: per-bin pooling without fbin_ptr");
  return ltm::pool_frames("frame pooling", k, dtype, xpart, a->Bv, a->L, a->T, a->e, binned ? 1 : splits, max_ctas,
                          stream, offs, frames, nullptr, 0, binned ? a->fbin_ptr : nullptr, a->xb_rows, ptrs);
}

// ------------------------------------------------------------------------------------------------
// One chunk of variant R for Bv videos:  pool -> (re-sample) -> consolidate -> project K,V ->
// continuous attention (+ next call's sticky histogram).  long_term_attention_gibbs.py:288-346.
// ------------------------------------------------------------------------------------------------
extern "C" int ltm_rect_step(const ltm_rect_step_args* a, const void* k, const float* q, const double* u,
                             const uint8_t* new_doc, float* ctx, void* stream) {
  using namespace ltm;
  LTM_REQUIRE(a && q && ctx, "rect_step: null pointer");
  if (int rc = check_chunk_dtype("rect_step", "k_dtype", a->k_dtype, a->e, a->binned != 0)) return rc;
  if (int rc = check_chunk_table("rect_step", "k_ptrs", a->k_ptrs, k, a->lengths, a->binned != 0)) return rc;
  const int D = a->H * a->d;
  const int qtiles = (a->Q + 31) / 32;
  cudaStream_t st_ = (cudaStream_t)stream;
#define LTM_PROF(i) do { if (a->prof_events[i]) cudaEventRecord((cudaEvent_t)a->prof_events[i], st_); } while (0)
  int rc = 0;
  const float* B_past = a->B_past;
  // binned: a->xpart carries per-bin sums of the pooled frames (ltm_pool_bins) and the update tables list bins
  const bool binned = a->binned != 0;
  if (binned) {
    LTM_REQUIRE(B_past != nullptr && new_doc == nullptr, "rect_step: bin sums only exist for update calls of all videos");
    LTM_REQUIRE(a->xb_rows > 0 && a->fbin_ptr && a->seg_ptr1b && a->seg_mem1b, "rect_step: binned tables missing");
  }
  // ragged batch: per-video lengths (0 = idle), tables from the bank, pooled frames packed by the frame offsets
  const int32_t* lengths = a->lengths;
  const bool ragged = lengths != nullptr;
  const size_t hist_bytes = sizeof(float) * a->H * qtiles * (LTM_STICKY_EDGES - 2);
  if (ragged) {
    LTM_REQUIRE(!binned, "rect_step: per-bin pooling does not apply to ragged batches");
    LTM_REQUIRE(a->frame_offs && a->bank_seg_ptr0 && a->bank_seg_mem0 && a->bank_g0 && a->bank_seg_ptr1 &&
                a->bank_seg_mem1 && a->bank_g1, "rect_step: ragged batch without frame offsets / table bank");
    LTM_REQUIRE(a->n_idle == 0 || !a->sticky || a->hist_keep, "rect_step: idle videos need hist_keep");
    if (a->n_idle > 0 && a->sticky) {
      rc = carry_idle(lengths, a->hist_part, a->hist_keep, hist_bytes, a->Bv, stream);
      if (rc) return rc;
    }
  }
  if (k != nullptr || a->k_ptrs != nullptr) {  // neither: a->xpart was already filled (frame pooling is stateless
    LTM_PROF(0);               // and may be issued ahead of time on another stream, see BatchedRectLTM.prefetch)
    rc = pool_chunk(a, k, a->k_ptrs, a->k_dtype, a->xpart, ragged ? a->frame_offs : nullptr, a->frames, a->splits, binned, 0,
                    stream);
    if (rc) return rc;
    LTM_PROF(1);
  }
  const int xL = binned ? a->xb_rows : a->L, xsplits = binned ? 1 : a->splits;
  const int32_t* seg_ptr0 = ragged ? a->bank_seg_ptr0 : a->seg_ptr0;
  const int32_t* seg_mem0 = ragged ? a->bank_seg_mem0 : a->seg_mem0;
  const float* g0 = ragged ? a->bank_g0 : a->g0;
  const int32_t* seg_ptr1 = ragged ? a->bank_seg_ptr1 : binned ? a->seg_ptr1b : a->seg_ptr1;
  const int32_t* seg_mem1 = ragged ? a->bank_seg_mem1 : binned ? a->seg_mem1b : a->seg_mem1;
  const float* g1 = ragged ? a->bank_g1 : a->g1;
  const int32_t* idx = a->idx_uniform;     // non-sticky: fixed table shared by all videos (index stride 0)
  long long idx_stride = 0;
  // (ragged: u == NULL when no video continues its memory in this call)
  if (B_past != nullptr && a->sticky && !(ragged && u == nullptr)) {
    LTM_REQUIRE(u != nullptr, "rect_step: sticky re-sampling needs the uniform draws");
    LTM_PROF(2);
    rc = ragged ? resample_ragged(a->hist_part, a->H * qtiles, LTM_STICKY_EDGES - 2, 1, u, a->bins, a->bin2basis, 0,
                                  a->p, a->b_draw, nullptr, a->ts, a->idx, a->Bv, a->S, lengths, stream)
                : ltm_resample(a->hist_part, a->H * qtiles, LTM_STICKY_EDGES - 2, 1, u, a->bins, a->bin2basis, 0, a->p,
                               a->b_draw, nullptr, a->ts, a->idx, a->Bv, a->S, stream);
    if (rc) return rc;
    LTM_PROF(3);
    idx = a->idx;
    idx_stride = a->S;
  }
  // tensor-core attention: row-major tf32-rounded K|V from the projection, both attention contractions as UMMAs
  const bool tc512 = a->attn_part != nullptr && a->scores != nullptr && ltm_attn_tc_split_supported(a->N, a->d);
  const bool tcp = a->X != nullptr && a->KV != nullptr && a->precision == 1 && a->gemm_impl == 0 &&
                   (ltm_attn_tc_supported(a->N, a->d) || tc512);
  const bool half_ops = tcp && a->B_half != nullptr && a->Wkv_half != nullptr && a->e % 8 == 0;
  const bool fast = !tcp && a->Kt != nullptr && a->V != nullptr && ltm_attn_fast_supported(a->N, a->d);
  // projected-memory state: every video updates, K|V of the previous call are at hand, and the rows that receive new
  // frames tile the 128-row GEMM tiles evenly -> only those rows are projected (row-major K|V layouts only)
  // (the projected rows start at jg <= jf, chosen so that N - jg divides -- or is a multiple of -- the 128-row GEMM
  // tile: bins in [jg, jf) hold re-sampled memory only and could go either way)
  int n_new = a->N - a->jf;
  if (n_new > 0 && n_new <= 128) {
    int p2 = 1;
    while (p2 < n_new) p2 <<= 1;
    n_new = p2;
  } else if (n_new > 128) {
    n_new = (n_new + 127) / 128 * 128;
  }
  const int jg = a->N - n_new;
  const bool kvstate = a->KV_past != nullptr && a->KV != nullptr && !fast && B_past != nullptr &&
                       new_doc == nullptr && a->jf > 0 && n_new > 0 && jg > 0 && a->e % 4 == 0;
  const int pprec = a->proj_precision ? a->proj_precision : a->precision;
  const bool kvh = a->kv_half != 0 && tcp && a->X16 != nullptr;                    // K|V stored as fp16
  const size_t sKV = (size_t)a->N * 2 * D;
  void* Bh = half_ops ? a->B_half : nullptr;
  LTM_PROF(4);
  rc = consolidate_rect_ragged(B_past, a->xpart, idx, idx_stride, new_doc, seg_ptr0, seg_mem0, g0, seg_ptr1, seg_mem1,
                               g1, a->B_new, Bh, kvstate ? a->KV_past : nullptr, a->KV, a->bkv, 2 * D, jg,
                               kvh ? 2 : (tcp ? 1 : 0), a->Bv, a->N, a->e, xL, xsplits, a->S,
                               ragged ? lengths : nullptr, ragged ? a->frame_offs : nullptr, stream);
  if (rc) return rc;
  LTM_PROF(5);
  LTM_PROF(6);
  // K|V projection KV = B_new W_kv^T + b_kv (fp16 operands: the fp16 copy of the new coefficient rows and of the
  // weights, kind::f16 UMMAs; K|V for the tensor-core attention is stored as fp16 or rounded to the tf32 grid)
  ltm_gemm_args ga;
  memset(&ga, 0, sizeof(ga));
  ga.A = half_ops ? reinterpret_cast<const float*>(Bh) : a->B_new; ga.lda = a->e; ga.a_kmajor = 1;
  ga.B = half_ops ? reinterpret_cast<const float*>(a->Wkv_half) : a->Wkv; ga.ldb = a->e; ga.b_kmajor = 1;
  ga.ab_fp16 = half_ops ? 1 : 0;
  ga.K1 = a->e; ga.bias = a->bkv;
  ga.C = a->KV; ga.ldc = 2 * D;
  ga.M = a->Bv * a->N; ga.Nc = 2 * D; ga.K = a->e; ga.batch = 1;
  // (the transposed-key and generic projections ignore proj_precision, except for the generic projected-memory rows)
  ga.precision = half_ops ? 1 : (tcp || kvstate) ? pprec : a->precision;
  ga.impl = a->gemm_impl; ga.round_tf32 = (tcp && !kvh) ? 1 : 0; ga.c_fp16 = kvh ? 1 : 0;
  // (only the fp16-operand, fp16-K|V and projected-memory projections take the grid bound)
  ga.max_ctas = (half_ops || kvh || kvstate) ? a->gemm_ctas : 0;
  if (kvstate) {
    // rows [jg, N) of every video as one flat problem: A = B_new + jg * e grouped per video, C = KV + jg * 2D
    ga.A = half_ops ? reinterpret_cast<const float*>(reinterpret_cast<const uint16_t*>(Bh) + (size_t)jg * a->e)
                    : a->B_new + (size_t)jg * a->e;
    ga.a_group = n_new; ga.a_group_stride = (int64_t)a->N * a->e;
    ga.C = kvh ? reinterpret_cast<float*>(reinterpret_cast<uint16_t*>(a->KV) + (size_t)jg * 2 * D)
               : a->KV + (size_t)jg * 2 * D;
    ga.c_group = n_new; ga.c_group_stride = (int64_t)a->N * 2 * D;
    ga.M = a->Bv * n_new;
  } else if (fast) {
    // keys transposed per head for the fast attention: Kt[Bv, H, d, N], values V[Bv, N, D]
    ga.C = a->V; ga.ldc = D;
    ga.CT = a->Kt; ga.ct_cols = D; ga.ct_group = a->N;
  }
  rc = ltm_gemm(&ga, stream);
  if (rc) return rc;
  LTM_PROF(7);
  LTM_PROF(8);
  float* hp = a->sticky ? a->hist_part : nullptr;
  if (kvh) {
    const uint16_t* Kh = reinterpret_cast<const uint16_t*>(a->KV);
    if (tc512)
      rc = ltm_cont_attn_rect_tc16_split(q, Kh, Kh + D, 2 * D, a->X16, a->W, a->W_out, a->jb, a->tb, ctx, a->scores,
                                         a->attn_part, hp, a->Bv, a->Q, a->N, a->H, a->d, stream);
    else
      rc = ltm_cont_attn_rect_tc16(q, Kh, Kh + D, 2 * D, a->X16, a->W, a->W_out, a->c_none, a->jb, a->tb, ctx,
                                   a->scores, hp, a->Bv, a->Q, a->N, a->H, a->d, stream);
  } else if (tcp && tc512)
    rc = ltm_cont_attn_rect_tc_split(q, a->KV, a->KV + D, 2 * D, a->X, a->W, a->W_out, a->jb, a->tb, ctx, a->scores,
                                     a->attn_part, hp, a->Bv, a->Q, a->N, a->H, a->d, stream);
  else if (tcp)
    rc = ltm_cont_attn_rect_tc(q, a->KV, a->KV + D, 2 * D, a->X, a->W, a->W_out, a->c_none, a->jb, a->tb, ctx,
                               a->scores, hp, a->Bv, a->Q, a->N, a->H, a->d, stream);
  else if (fast)
    rc = ltm_cont_attn_rect_t(q, a->Kt, a->V, D, a->W, a->W_out, a->jb, a->tb, ctx, a->scores, hp, a->Bv, a->Q, a->N,
                              a->H, a->d, stream);
  else
    rc = ltm_cont_attn_rect(q, a->KV, a->W, a->W_out, a->jb, a->tb, ctx, a->scores, hp, a->Bv, a->Q, a->N, a->H, a->d,
                            stream);
  if (rc) return rc;
  LTM_PROF(9);
#undef LTM_PROF
  if (ragged && a->n_idle > 0) {
    // idle videos: the consolidation copied their coefficients into B_new, and the projection and attention ran over
    // them; what those overwrote goes back to what it was -- the carried K|V into the buffer of the next call, the saved
    // histogram partials -- and their context rows are zero.  (Without KV_past the K|V rows just projected from the
    // kept coefficients stay.)
    if (a->KV_past && a->KV) rc = carry_idle(lengths, a->KV_past, a->KV, (kvh ? 2 : 4) * sKV, a->Bv, stream);
    if (!rc && a->sticky) rc = carry_idle(lengths, a->hist_keep, a->hist_part, hist_bytes, a->Bv, stream);
    if (!rc) rc = carry_idle(lengths, nullptr, ctx, sizeof(float) * a->Q * D, a->Bv, stream);
  }
  return rc;
}

extern "C" int ltm_rect_step_overlap(const ltm_rect_step_args* a, const ltm_overlap* o, const float* q,
                                     const double* u, const uint8_t* new_doc, float* ctx) {
  using namespace ltm;
  LTM_REQUIRE(a && o && q && ctx, "rect_step_overlap: null pointer");
  LTM_REQUIRE(o->ev_fork && o->ev_join, "rect_step_overlap: fork / join events missing");
  if (int rc = check_chunk_dtype("rect_step_overlap", "k_dtype", a->k_dtype, a->e, a->binned != 0)) return rc;
  if (int rc = check_chunk_table("rect_step_overlap", "k_ptrs", a->k_ptrs, nullptr, a->lengths, a->binned != 0))
    return rc;
  if (int rc = check_chunk_table("rect_step_overlap", "next_ptrs", o->next_ptrs, o->k_next, o->next_lengths,
                                 o->next_binned != 0))
    return rc;
  const bool pool_next = o->k_next != nullptr || o->next_ptrs != nullptr;
  if (pool_next) {
    if (int rc = check_chunk_dtype("rect_step_overlap", "next_dtype", o->next_dtype, a->e, o->next_binned != 0))
      return rc;
    LTM_REQUIRE(o->xpart_next && o->ev_fork_pool && o->ev_pooled_next, "rect_step_overlap: prefetch target missing");
    LTM_REQUIRE(!o->next_lengths || (o->next_offs && !o->next_binned), "rect_step_overlap: ragged next chunk");
  }
  cudaStream_t ms = (cudaStream_t)o->main_stream, ss = (cudaStream_t)o->side_stream,
               cs = (cudaStream_t)o->compute_stream;
  if (pool_next) {
    // the target buffer was last read by work already queued on the main stream
    LTM_CUDA(cudaEventRecord((cudaEvent_t)o->ev_fork_pool, ms));
    LTM_CUDA(cudaStreamWaitEvent(ss, (cudaEvent_t)o->ev_fork_pool, 0));
    if (a->prof_events[0]) cudaEventRecord((cudaEvent_t)a->prof_events[0], ss);
    const bool ragged_next = o->next_lengths != nullptr;
    int rc = pool_chunk(a, o->k_next, o->next_ptrs, o->next_dtype, o->xpart_next, ragged_next ? o->next_offs : nullptr,
                        o->next_frames, ragged_next ? o->next_splits : a->splits, o->next_binned != 0, o->pool_ctas,
                        ss);
    if (rc) return rc;
    if (a->prof_events[1]) cudaEventRecord((cudaEvent_t)a->prof_events[1], ss);
    LTM_CUDA(cudaEventRecord((cudaEvent_t)o->ev_pooled_next, ss));
  }
  LTM_CUDA(cudaEventRecord((cudaEvent_t)o->ev_fork, ms));
  LTM_CUDA(cudaStreamWaitEvent(cs, (cudaEvent_t)o->ev_fork, 0));
  if (o->ev_pooled_cur) LTM_CUDA(cudaStreamWaitEvent(cs, (cudaEvent_t)o->ev_pooled_cur, 0));
  int rc = ltm_rect_step(a, nullptr, q, u, new_doc, ctx, cs);
  if (rc) return rc;
  LTM_CUDA(cudaEventRecord((cudaEvent_t)o->ev_join, cs));
  LTM_CUDA(cudaStreamWaitEvent(ms, (cudaEvent_t)o->ev_join, 0));
  return 0;
}

extern "C" int ltm_event_create(void** ev) {
  using namespace ltm;
  LTM_REQUIRE(ev != nullptr, "event_create: null pointer");
  cudaEvent_t e;
  LTM_CUDA(cudaEventCreate(&e));
  *ev = (void*)e;
  return 0;
}
extern "C" int ltm_event_create_sync(void** ev) {
  using namespace ltm;
  LTM_REQUIRE(ev != nullptr, "event_create_sync: null pointer");
  cudaEvent_t e;
  LTM_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  *ev = (void*)e;
  return 0;
}
extern "C" int ltm_stream_wait_event(void* stream, void* ev) {
  using namespace ltm;
  LTM_CUDA(cudaStreamWaitEvent((cudaStream_t)stream, (cudaEvent_t)ev, 0));
  return 0;
}
extern "C" int ltm_event_record(void* ev, void* stream) {
  using namespace ltm;
  LTM_CUDA(cudaEventRecord((cudaEvent_t)ev, (cudaStream_t)stream));
  return 0;
}
extern "C" int ltm_event_elapsed_ms(void* start, void* stop, float* ms) {
  using namespace ltm;
  LTM_REQUIRE(ms != nullptr, "event_elapsed_ms: null pointer");
  cudaError_t e = cudaEventSynchronize((cudaEvent_t)stop);
  if (e == cudaSuccess) e = cudaEventElapsedTime(ms, (cudaEvent_t)start, (cudaEvent_t)stop);
  if (e != cudaSuccess) {
    (void)cudaGetLastError();            // e.g. an event that was never recorded: do not leave a stale error behind
    set_error("event_elapsed_ms: %s", cudaGetErrorString(e));
    return -3;
  }
  return 0;
}
extern "C" int ltm_event_destroy(void* ev) {
  using namespace ltm;
  LTM_CUDA(cudaEventDestroy((cudaEvent_t)ev));
  return 0;
}

extern "C" int ltm_rect_step_host(const ltm_rect_step_args* a, const void* k_host, const float* q_host,
                                  const double* u_host, const uint8_t* new_doc_host, float* ctx_host, void* stream) {
  using namespace ltm;
  LTM_REQUIRE(a && k_host && q_host && ctx_host, "rect_step_host: null pointer");
  LTM_REQUIRE(a->k_dev && a->q_dev && a->ctx_dev, "rect_step_host: device staging buffers missing");
  if (int rc = check_chunk_dtype("rect_step_host", "k_dtype", a->k_dtype, a->e, a->binned != 0)) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const size_t D = (size_t)a->H * a->d;
  const size_t elem = a->k_dtype ? 2 : 4;           // k_host and k_dev hold the chunk in its own storage
  LTM_CUDA(cudaMemcpyAsync(a->k_dev, k_host, elem * (size_t)a->Bv * a->L * a->T * a->e, cudaMemcpyHostToDevice, st));
  LTM_CUDA(cudaMemcpyAsync(a->q_dev, q_host, sizeof(float) * (size_t)a->Bv * a->Q * D, cudaMemcpyHostToDevice, st));
  const double* u_dev = nullptr;
  if (u_host) {
    LTM_REQUIRE(a->u_dev, "rect_step_host: u staging buffer missing");
    LTM_CUDA(cudaMemcpyAsync(a->u_dev, u_host, sizeof(double) * (size_t)a->Bv * a->S, cudaMemcpyHostToDevice, st));
    u_dev = a->u_dev;
  }
  const uint8_t* nd_dev = nullptr;
  if (new_doc_host) {
    LTM_REQUIRE(a->new_doc_dev, "rect_step_host: new_doc staging buffer missing");
    LTM_CUDA(cudaMemcpyAsync(a->new_doc_dev, new_doc_host, (size_t)a->Bv, cudaMemcpyHostToDevice, st));
    nd_dev = a->new_doc_dev;
  }
  int rc = ltm_rect_step(a, a->k_dev, a->q_dev, u_dev, nd_dev, a->ctx_dev, stream);
  if (rc) return rc;
  LTM_CUDA(cudaMemcpyAsync(ctx_host, a->ctx_dev, sizeof(float) * (size_t)a->Bv * a->Q * D, cudaMemcpyDeviceToHost, st));
  return 0;
}
