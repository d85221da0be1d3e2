"""Python wrappers of the individual libinfltm kernels (one per row of include/infltm.h).

Every function takes/returns CUDA tensors, launches on torch's current stream and never synchronises.
torch is used for device memory and streams only; all arithmetic happens in libinfltm.so."""
import ctypes as C

import torch

from . import _capi
from ._capi import GemmArgs, check, lib, ptr, require_cuda, stream_ptr

STICKY_EDGES = 129
PRECISION = {"tf32": 1, "tf32x3": 3, 1: 1, 3: 3}
GEMM_IMPL = {"tcgen05": 0, "simt": 1, 0: 0, 1: 1}


def _f32c(t):
    if t.dtype != torch.float32:
        raise ValueError(f"expected float32, got {t.dtype}")
    return t if t.is_contiguous() else t.contiguous()


def _rowmajor(t):
    """float32 2-D/3-D operand whose rows are dense (row pitch may exceed the row length)."""
    if t.dtype != torch.float32:
        raise ValueError(f"expected float32, got {t.dtype}")
    if t.stride(-1) != 1 or (t.dim() == 3 and t.shape[0] > 1 and t.stride(0) < t.stride(1)):
        t = t.contiguous()
    return t


# storage of a chunk k as the library takes it (ltm_rect_step_args.k_dtype, ltm_overlap.next_dtype)
CHUNK_DTYPES = {torch.float32: 0, torch.float16: 1, torch.bfloat16: 2}


def pool_into(k, out, L, T, splits, max_ctas=0, stream=None, offs=None, frames=0, fbin_ptr=None, rows=0):
    """Frame pooling of a contiguous chunk k of Bv videos of L frames of T tokens of width e (float32 / float16 /
    bfloat16) into `out`, on `stream` (default: torch's current stream).  With offs (int32 [Bv+1] device frame
    offsets, `frames` in all): the packed frames of a ragged chunk, [frames, splits, e].  With fbin_ptr (float32
    chunks, tables.RectTables.fbin_ptr): the per-bin sums of an update chunk, [Bv, rows, e].  Otherwise the frame
    means as `splits` partial sums, [Bv, L, splits, e].  max_ctas > 0 bounds the grid (0: one CTA per frame-split)."""
    Bv, e = k.shape[0], k.shape[-1]
    dt = CHUNK_DTYPES[k.dtype]
    st = stream_ptr(k.device) if stream is None else stream
    if offs is not None:
        check(lib().ltm_pool_mean_ragged(ptr(k), dt, ptr(out), ptr(offs), Bv, L, T, e, splits, frames, max_ctas, st),
              "pool_mean_ragged")
    elif fbin_ptr is not None:
        check(lib().ltm_pool_bins(ptr(k), ptr(out), ptr(fbin_ptr), Bv, L, T, e, rows, st), "pool_bins")
    elif dt:
        check(lib().ltm_pool_mean_16_grid(ptr(k), int(dt == 2), ptr(out), Bv, L, T, e, splits, max_ctas, st),
              "pool_mean_16_grid")
    else:
        check(lib().ltm_pool_mean_grid(ptr(k), ptr(out), Bv, L, T, e, splits, max_ctas, st), "pool_mean")


def pool_ptrs(ptrs, dtype, out, offs, Bv, L, T, e, splits, frames, max_ctas=0, stream=None):
    """`pool_into` of a ragged chunk whose videos live at their own addresses: ptrs int64 [Bv] device table of base
    addresses (video v's lengths[v]*T dense rows of width e, 16-byte aligned; idle videos are not read), dtype a
    `CHUNK_DTYPES` code, offs int32 [Bv+1] device frame offsets -> out[frames, splits, e] (any float32 storage of that
    many elements), bit for bit what `pool_into` gives with offs for the same frames of a padded chunk."""
    require_cuda(ptrs, out, offs)
    st = stream_ptr(out.device) if stream is None else stream
    check(lib().ltm_pool_mean_ptrs(ptr(ptrs), dtype, ptr(out), ptr(offs), Bv, L, T, e, splits, frames, max_ctas, st),
          "pool_mean_ptrs")


def pool_mean(k, splits=1):
    """k[Bv,L,T,e] -> xpart[Bv,L,splits,e] (frame means as `splits` partial sums).  gibbs:304."""
    require_cuda(k)
    Bv, L, T, e = k.shape
    out = torch.empty(Bv, L, splits, e, device=k.device, dtype=torch.float32)
    # a 16-bit chunk is read as is and accumulated in fp32
    k = k.contiguous() if k.dtype in (torch.float16, torch.bfloat16) else _f32c(k)
    pool_into(k, out, L, T, splits)
    return out


def pool_mean_convert(k, splits=1):
    """`pool_mean` that also returns the chunk as float16: k[Bv,L,T,e] fp32 -> (xpart[Bv,L,splits,e], k16[Bv,L,T,e])."""
    require_cuda(k)
    k = _f32c(k)
    Bv, L, T, e = k.shape
    out = torch.empty(Bv, L, splits, e, device=k.device, dtype=torch.float32)
    k16 = torch.empty(Bv, L, T, e, device=k.device, dtype=torch.float16)
    check(lib().ltm_pool_mean_convert(ptr(k), ptr(out), ptr(k16), Bv, L, T, e, splits, stream_ptr(k.device)),
          "pool_mean_convert")
    return out, k16


def pool_mean_convert_ragged(k, offs, frames, splits, ld16):
    """Ragged `pool_mean_convert`: k[Bv,L,T,e] fp32 padded, offs int32 [Bv+1] device frame offsets (exclusive prefix sum
    of the lengths, `frames` = offs[Bv]) -> (xpart[frames, splits, e] packed video after video, k16[Bv, ld16, e]).
    k16 rows [0, n_v) of video v hold its first lengths[v] * T tokens as fp16, rows [n_v, roundup64(n_v)) are zero and
    the rest is left unwritten (ld16 % 64 == 0, ld16 >= L*T)."""
    require_cuda(k, offs)
    k = _f32c(k)
    Bv, L, T, e = k.shape
    out = torch.empty(frames, splits, e, device=k.device, dtype=torch.float32)
    k16 = torch.empty(Bv, ld16, e, device=k.device, dtype=torch.float16)
    check(lib().ltm_pool_mean_convert_ragged(ptr(k), ptr(out), ptr(k16), ptr(offs), Bv, L, T, e, splits, frames, ld16,
                                             stream_ptr(k.device)), "pool_mean_convert_ragged")
    return out, k16


def pool_bins(k, fbin_ptr, rows):
    """Per-bin pooling of an update chunk: k[Bv,L,T,e] fp32, fbin_ptr int32 [rows+1] -> xbin[Bv,rows,e], the sum of the
    pooled frames [fbin_ptr[r], fbin_ptr[r+1]) (tables.RectTables.fbin_ptr)."""
    require_cuda(k, fbin_ptr)
    k = _f32c(k)
    Bv, L, T, e = k.shape
    out = torch.empty(Bv, rows, e, device=k.device, dtype=torch.float32)
    pool_into(k, out, L, T, 1, fbin_ptr=fbin_ptr, rows=rows)
    return out


def consolidate_rect_kv(B_past, xpart, idx, tab, S, KV_past, bkv, jf, round_tf32=False, new_doc=None):
    """`consolidate_rect` that also carries the projected memory K|V along: rows j < jf of KV_new are the segmented
    mean of KV_past rows (+ bias term); rows >= jf are left untouched for the projection GEMM.  idx: [Bv,S] or [S]
    (one row shared by all videos).  Returns (B_new, KV_new)."""
    require_cuda(B_past, xpart, idx, KV_past, bkv, new_doc)
    Bv, L, splits, e = xpart.shape
    N = tab["g0"].numel()
    ldkv = KV_past.shape[-1]
    B_new = torch.empty(Bv, N, e, device=xpart.device, dtype=torch.float32)
    KV_new = torch.zeros(Bv, N, ldkv, device=xpart.device, dtype=torch.float32)
    check(lib().ltm_consolidate_rect_kv(ptr(B_past), ptr(xpart), ptr(idx), S if idx.dim() == 2 else 0, ptr(new_doc),
                                        ptr(tab["seg_ptr0"]), ptr(tab["seg_mem0"]), ptr(tab["g0"]),
                                        ptr(tab["seg_ptr1"]), ptr(tab["seg_mem1"]), ptr(tab["g1"]),
                                        ptr(B_new), None, ptr(KV_past), ptr(KV_new), ptr(bkv), ldkv, jf,
                                        int(bool(round_tf32)), Bv, N, e, L, splits, S, stream_ptr(xpart.device)),
          "consolidate_rect_kv")
    return B_new, KV_new


def kl_gauss(mu, sd, mu_0, sigma_0):
    """KL regulariser of the Gaussian variant per (video, head*query) row (long_term_attention.py:296-304)."""
    require_cuda(mu, sd)
    mu, sd = _f32c(mu), _f32c(sd)
    out = torch.empty_like(mu)
    check(lib().ltm_kl_gauss(ptr(mu), ptr(sd), float(mu_0), float(sigma_0), ptr(out), mu.numel(),
                             stream_ptr(mu.device)), "kl_gauss")
    return out


def sticky_hist_rect(scores, jb, tb):
    """scores[Bv,H,Q,N] -> hist_part[Bv,H,127].  gibbs:196-203."""
    require_cuda(scores, jb, tb)
    scores = _f32c(scores)
    Bv, H, Q, N = scores.shape
    out = torch.empty(Bv, H, STICKY_EDGES - 2, device=scores.device, dtype=torch.float32)
    check(lib().ltm_sticky_hist_rect(ptr(scores), ptr(jb), ptr(tb), ptr(out), Bv, H, Q, N,
                                     stream_ptr(scores.device)), "sticky_hist_rect")
    return out


def density_rect(scores, jd, wd):
    """scores[Bv,H,Q,N] -> alphas[Q,Bv,H,768] (density side-output of the Video-LLaMA copy, gibbs:320-343)."""
    require_cuda(scores, jd, wd)
    scores = _f32c(scores)
    Bv, H, Q, N = scores.shape
    out = torch.empty(Q, Bv, H, 768, device=scores.device, dtype=torch.float32)
    check(lib().ltm_density_rect(ptr(scores), ptr(jd), ptr(wd), ptr(out), Bv, H, Q, N, stream_ptr(scores.device)),
          "density_rect")
    return out


def sticky_hist_gauss(mu, sd, tb, parts=None):
    """mu,sd[Bv,R] -> hist_part[Bv,parts,128] (feed to `resample`).  long_term_attention.py:220-229."""
    require_cuda(mu, sd, tb)
    mu, sd = _f32c(mu), _f32c(sd)
    Bv, R = mu.shape
    if parts is None:
        parts = max(1, min(8, R // 48))          # ~48 rows per CTA: 8 CTAs per video at R = H*Q = 384
    out = torch.empty(Bv, parts, STICKY_EDGES - 1, device=mu.device, dtype=torch.float32)
    check(lib().ltm_sticky_hist_gauss(ptr(mu), ptr(sd), ptr(tb), ptr(out), Bv, R, parts, stream_ptr(mu.device)),
          "sticky_hist_gauss")
    return out


def resample(hist_part, u, bins, bin2basis=None, normalize=True, sort=False, out=None):
    """Inverse-CDF sampling with explicit fp64 uniforms.  hist_part[Bv,parts,ncat] (or [Bv,ncat]),
    u[Bv,S] -> dict(p, b_draw, b_used, ts, idx).  gibbs:204-208 / gauss:230-238."""
    require_cuda(hist_part, u, bins, bin2basis)
    hist_part = _f32c(hist_part)
    if hist_part.dim() == 2:
        hist_part = hist_part.unsqueeze(1)
    Bv, parts, ncat = hist_part.shape
    if u.dtype != torch.float64 or u.shape[0] != Bv:
        raise ValueError("u must be float64 [Bv,S]")
    u = u.contiguous()
    S = u.shape[1]
    dev = hist_part.device
    o = out or {}
    o.setdefault("p", torch.empty(Bv, ncat, device=dev, dtype=torch.float32))
    for name in ("b_draw", "b_used", "idx"):
        o.setdefault(name, torch.empty(Bv, S, device=dev, dtype=torch.int32))
    o.setdefault("ts", torch.empty(Bv, S, device=dev, dtype=torch.float32))
    check(lib().ltm_resample(ptr(hist_part), parts, ncat, int(bool(normalize)), ptr(u), ptr(bins), ptr(bin2basis),
                             int(bool(sort)), ptr(o["p"]), ptr(o["b_draw"]), ptr(o["b_used"]), ptr(o["ts"]),
                             ptr(o["idx"]), Bv, S, stream_ptr(dev)), "resample")
    return o


def consolidate_rect(B_past, xpart, idx, new_doc, tab, S, out=None):
    """Segmented-mean regression of variant R.  `tab` = RectTables.to(device).  gibbs:184-222."""
    require_cuda(B_past, xpart, idx, new_doc)
    Bv, L, splits, e = xpart.shape
    N = tab["g0"].numel()
    if out is None:
        out = torch.empty(Bv, N, e, device=xpart.device, dtype=torch.float32)
    check(lib().ltm_consolidate_rect(ptr(B_past), ptr(xpart), ptr(idx), ptr(new_doc),
                                     ptr(tab["seg_ptr0"]), ptr(tab["seg_mem0"]), ptr(tab["g0"]),
                                     ptr(tab["seg_ptr1"]), ptr(tab["seg_mem1"]), ptr(tab["g1"]),
                                     ptr(out), Bv, N, e, L, splits, S, stream_ptr(xpart.device)),
          "consolidate_rect")
    return out


def gemm(A, B, *, a_kmajor=True, b_kmajor=True, B2=None, bias=None, out=None, precision="tf32x3",
         impl="tcgen05", M=None, Nc=None, K=None):
    """Batched C[b] = A[b] @ B[b] (+bias) on tcgen05 (kind::tf32).

    A: [batch?, M, K] if a_kmajor else [batch?, K, M];  B: [batch?, Nc, K] if b_kmajor else [batch?, K, Nc].
    A 2-D operand is shared by every batch.  B2 (same layout as B) continues B along K."""
    require_cuda(A, B, B2, bias, out)
    A, B = _rowmajor(A), _rowmajor(B)
    batch = max(A.shape[0] if A.dim() == 3 else 1, B.shape[0] if B.dim() == 3 else 1)

    def desc(t, kmajor):
        m = t if t.dim() == 3 else t.unsqueeze(0)
        stride = m.stride(0) if (t.dim() == 3 and t.shape[0] > 1) else 0
        rows, k = (m.shape[1], m.shape[2]) if kmajor else (m.shape[2], m.shape[1])
        return rows, k, m.stride(1), stride

    Ma, Ka, lda, sA = desc(A, a_kmajor)
    Nb, Kb, ldb, sB = desc(B, b_kmajor)
    if A.dim() == 3 and A.shape[0] == batch and batch > 1:
        sA = A.stride(0)
    if B.dim() == 3 and B.shape[0] == batch and batch > 1:
        sB = B.stride(0)
    K1 = Kb
    ldb2 = sB2 = 0
    if B2 is not None:
        B2 = _rowmajor(B2)
        Nb2, Kb2, ldb2, sB2 = desc(B2, b_kmajor)
        if B2.dim() == 3 and B2.shape[0] == batch and batch > 1:
            sB2 = B2.stride(0)
        if Nb2 != Nb:
            raise ValueError("B and B2 disagree on N")
        Kb = Kb + Kb2
    if Ka != Kb:
        raise ValueError(f"inner dimensions disagree: A has K={Ka}, B has K={Kb}")
    M = Ma if M is None else M
    Nc = Nb if Nc is None else Nc
    if out is None:
        out = torch.empty(batch, M, Nc, device=A.device, dtype=torch.float32)
    o3 = out if out.dim() == 3 else out.unsqueeze(0)
    g = GemmArgs()
    g.A, g.lda, g.strideA, g.a_kmajor = A.data_ptr(), lda, sA, int(a_kmajor)
    g.B, g.ldb, g.strideB, g.b_kmajor = B.data_ptr(), ldb, sB, int(b_kmajor)
    g.B2 = B2.data_ptr() if B2 is not None else None
    g.ldb2, g.strideB2, g.K1 = ldb2, sB2, K1
    g.bias = bias.data_ptr() if bias is not None else None
    g.C, g.ldc, g.strideC = o3.data_ptr(), o3.stride(1), (o3.stride(0) if batch > 1 else 0)
    g.M, g.Nc, g.K, g.batch = M, Nc, Ka, batch
    g.precision, g.impl = PRECISION[precision], GEMM_IMPL[impl]
    g.CT, g.ct_cols, g.ct_group = None, 0, 0
    check(lib().ltm_gemm(C.byref(g), stream_ptr(A.device)), "gemm")
    return out


def gemm_raw(A, lda, strideA, a_kmajor, B, ldb, strideB, b_kmajor, C_, ldc, strideC, M, Nc, K, batch, *, bias=None,
             bias_stride=0, c_group=0, c_group_stride=0, precision="tf32", impl="tcgen05", a_offset=0, b_offset=0,
             c_offset=0, round_tf32=False, a_group=0, a_group_stride=0, bias_offset=0, c_fp16=False, ab_fp16=False,
             C_lo=None, max_ctas=0, n_ext=None, k_ext=None):
    """ltm_gemm with every pitch / batch stride spelled out (elements).  A, B, C_ are the base tensors; *_offset
    shifts the start (elements).  Used where operands are strided views that tensor shapes cannot express
    (per-head column blocks, per-head / per-video output layouts).
    n_ext / k_ext: optional contiguous device int32 [batch] extents (ltm_gemm_extents, fp16 operands only): tiles of
    batch b starting at column >= n_ext[b] are skipped, batch b runs k_ext[b] (a multiple of 64) K-elements; a batch
    with an extent of 0 leaves its C unwritten."""
    require_cuda(A, B, C_, bias, n_ext, k_ext)
    for ext in (n_ext, k_ext):
        if ext is not None and (ext.dtype != torch.int32 or not ext.is_contiguous() or ext.numel() != batch):
            raise ValueError(f"gemm extents must be contiguous int32 tensors of {batch} entries")
    g = GemmArgs()
    esz = 2 if ab_fp16 else 4                     # (ab_fp16: A and B are float16 tensors, offsets in elements)
    g.A, g.lda, g.strideA, g.a_kmajor = A.data_ptr() + esz * a_offset, lda, strideA, int(a_kmajor)
    g.B, g.ldb, g.strideB, g.b_kmajor = B.data_ptr() + esz * b_offset, ldb, strideB, int(b_kmajor)
    g.ab_fp16 = int(bool(ab_fp16))
    g.B2, g.ldb2, g.strideB2, g.K1 = None, 0, 0, K
    g.bias = bias.data_ptr() + 4 * bias_offset if bias is not None else None
    g.bias_stride = bias_stride
    g.C, g.ldc, g.strideC = C_.data_ptr() + (2 if c_fp16 else 4) * c_offset, ldc, strideC
    g.c_fp16 = int(bool(c_fp16))
    g.C_lo = (C_lo.data_ptr() + 2 * c_offset) if C_lo is not None else None      # residual fp16 term (c_fp16 only)
    g.max_ctas = int(max_ctas)                    # bound of the persistent grid (0 = one CTA per SM)
    g.M, g.Nc, g.K, g.batch = M, Nc, K, batch
    g.precision, g.impl = PRECISION[precision], GEMM_IMPL[impl]
    g.CT, g.ct_cols, g.ct_group = None, 0, 0
    g.c_group, g.c_group_stride = c_group, c_group_stride
    g.round_tf32 = int(bool(round_tf32))
    g.a_group, g.a_group_stride = a_group, a_group_stride
    if n_ext is not None or k_ext is not None:
        check(lib().ltm_gemm_extents(C.byref(g), ptr(n_ext), ptr(k_ext), stream_ptr(A.device)), "gemm_extents")
        return C_
    check(lib().ltm_gemm(C.byref(g), stream_ptr(A.device)), "gemm")
    return C_


def gemm_fp16(A, B, bias=None, out=None, round_tf32=False):
    """C[M,Nc] fp32 = A[M,K] fp16 @ B[Nc,K]^T fp16 (+ bias): kind::f16 UMMAs, fp32 accumulation (`ab_fp16`)."""
    require_cuda(A, B, bias)
    if A.dtype != torch.float16 or B.dtype != torch.float16 or not A.is_contiguous() or not B.is_contiguous():
        raise ValueError("gemm_fp16 takes contiguous float16 operands")
    M, K = A.shape
    Nc = B.shape[0]
    if out is None:
        out = torch.empty(M, Nc, device=A.device, dtype=torch.float32)
    g = GemmArgs()
    g.A, g.lda, g.strideA, g.a_kmajor = A.data_ptr(), K, 0, 1
    g.B, g.ldb, g.strideB, g.b_kmajor = B.data_ptr(), K, 0, 1
    g.B2, g.ldb2, g.strideB2, g.K1 = None, 0, 0, K
    g.bias = bias.data_ptr() if bias is not None else None
    g.C, g.ldc, g.strideC = out.data_ptr(), Nc, 0
    g.M, g.Nc, g.K, g.batch = M, Nc, K, 1
    g.precision, g.impl = 1, 0
    g.round_tf32, g.ab_fp16 = int(bool(round_tf32)), 1
    check(lib().ltm_gemm(C.byref(g), stream_ptr(A.device)), "gemm(fp16)")
    return out


def _check_softmax_mask(S, mask, rows, n, rows_per_mask, what):
    """The kernels read mask row `row // rows_per_mask` at pitch n, unchecked: the mask must hold exactly those rows."""
    if mask is None:
        return
    if mask.dtype != torch.float32 or not mask.is_contiguous() or mask.device != S.device:
        raise ValueError(f"{what}: the mask must be a contiguous float32 tensor on {S.device}, got {mask.dtype} "
                         f"on {mask.device}")
    if rows_per_mask <= 0 or rows % rows_per_mask:
        raise ValueError(f"{what}: rows_per_mask={rows_per_mask} must divide rows={rows}")
    if mask.numel() != (rows // rows_per_mask) * n:
        raise ValueError(f"{what}: the mask has {mask.numel()} elements, {rows // rows_per_mask} rows of {n} expected")


def softmax_rows(S, scale=1.0, mask=None, rows_per_mask=1):
    """In place: S[rows, n] <- softmax(S * scale + mask[row // rows_per_mask]).  Qformer.py:279-285."""
    require_cuda(S, mask)
    if not S.is_contiguous() or S.dtype != torch.float32:
        raise ValueError("softmax_rows needs a contiguous float32 tensor")
    n = S.shape[-1]
    rows = S.numel() // n
    _check_softmax_mask(S, mask, rows, n, rows_per_mask, "softmax_rows")
    check(lib().ltm_softmax_rows(ptr(S), ptr(mask), rows, n, rows_per_mask, float(scale), stream_ptr(S.device)),
          "softmax_rows")
    return S


def softmax_rows_half(S, scale=1.0, mask=None, rows_per_mask=1):
    """softmax(S * scale + mask) with the probabilities returned as float16 (S is scratch afterwards)."""
    require_cuda(S, mask)
    if not S.is_contiguous() or S.dtype != torch.float32:
        raise ValueError("softmax_rows_half needs a contiguous float32 tensor")
    n = S.shape[-1]
    rows = S.numel() // n
    _check_softmax_mask(S, mask, rows, n, rows_per_mask, "softmax_rows_half")
    P = torch.empty(S.shape, device=S.device, dtype=torch.float16)
    check(lib().ltm_softmax_rows_h(ptr(S), ptr(mask), ptr(P), rows, n, rows_per_mask, float(scale),
                                   stream_ptr(S.device)), "softmax_rows_h")
    return P


def softmax_rows_half_len(S, n_len, rows_per_len, scale=1.0, mask=None):
    """Ragged `softmax_rows_half`: S[..., ld] fp32 (ld % 64 == 0), n_len device int32 [rows / rows_per_len]: row r spans
    the first n_len[r // rows_per_len] <= ld columns.  Returns P fp16 of S's shape: softmax(S * scale + mask) on those
    columns, zeros up to the next multiple of 64, the rest unwritten (rows with n = 0 entirely).  mask: float32 rows
    [rows / rows_per_len, mask_ld] (only their first n columns are read) or None."""
    require_cuda(S, n_len, mask)
    if not S.is_contiguous() or S.dtype != torch.float32:
        raise ValueError("softmax_rows_half_len needs a contiguous float32 tensor")
    ld = S.shape[-1]
    rows = S.numel() // ld
    if rows_per_len <= 0 or rows % rows_per_len:
        raise ValueError(f"softmax_rows_half_len: rows_per_len={rows_per_len} must divide rows={rows}")
    if n_len.dtype != torch.int32 or not n_len.is_contiguous() or n_len.numel() != rows // rows_per_len:
        raise ValueError(f"softmax_rows_half_len: n_len must be contiguous int32 with {rows // rows_per_len} entries")
    mask_ld = 0
    if mask is not None:
        if mask.dtype != torch.float32 or not mask.is_contiguous() or mask.device != S.device or mask.dim() != 2 \
                or mask.shape[0] != rows // rows_per_len:
            raise ValueError(f"softmax_rows_half_len: the mask must be contiguous float32 [{rows // rows_per_len}, n] "
                             f"on {S.device}")
        mask_ld = mask.shape[1]
    P = torch.empty(S.shape, device=S.device, dtype=torch.float16)
    check(lib().ltm_softmax_rows_h_len(ptr(S), ptr(mask), ptr(P), ptr(n_len), rows, ld, mask_ld, rows_per_len,
                                       float(scale), stream_ptr(S.device)), "softmax_rows_h_len")
    return P


def to_half(x):
    """fp32 -> fp16 copy (round to nearest even) by the library's streaming kernel."""
    require_cuda(x)
    x = _f32c(x)
    out = torch.empty(x.shape, device=x.device, dtype=torch.float16)
    check(lib().ltm_to_half(ptr(x), ptr(out), x.numel(), stream_ptr(x.device)), "to_half")
    return out


def blend(a, b, alpha, out=None):
    """out = alpha * a + (1 - alpha) * b.  Qformer.py:303-304."""
    require_cuda(a, b)
    a, b = _f32c(a), _f32c(b)
    if out is None:
        out = torch.empty_like(a)
    check(lib().ltm_blend(ptr(a), ptr(b), float(alpha), ptr(out), a.numel(), stream_ptr(a.device)), "blend")
    return out


def project_kv(Bcoef, Wkv, bkv, precision="tf32", impl="tcgen05", out=None):
    """KV[M,2D] = Bcoef[M,e] @ Wkv[2D,e]^T + bkv.  gibbs:312-313."""
    require_cuda(Bcoef, Wkv, bkv)
    Bc = _f32c(Bcoef).reshape(-1, Bcoef.shape[-1])
    M, e = Bc.shape
    D2 = Wkv.shape[0]
    if out is None:
        out = torch.empty(M, D2, device=Bc.device, dtype=torch.float32)
    check(lib().ltm_project_kv(ptr(Bc), ptr(Wkv), ptr(bkv), ptr(out), M, e, D2, PRECISION[precision],
                               GEMM_IMPL[impl], stream_ptr(Bc.device)), "project_kv")
    return out


def attn_fast_supported(N, d=64):
    return bool(lib().ltm_attn_fast_supported(int(N), int(d)))


def attn_tc_supported(N, d=64):
    return bool(lib().ltm_attn_tc_supported(int(N), int(d)))


def attn_tc_split_supported(N, d=64):
    """num_basis 512: the tensor-core attention in two basis halves + combine (ltm_cont_attn_rect_tc_split)."""
    return bool(lib().ltm_attn_tc_split_supported(int(N), int(d)))


def project_kv_r(Bcoef, Wkv, bkv, precision="tf32", out=None):
    """`project_kv` with the stored K|V rounded to the tf32 grid (operands of the tensor-core attention)."""
    require_cuda(Bcoef, Wkv, bkv)
    Bc = _f32c(Bcoef).reshape(-1, Bcoef.shape[-1])
    M, e = Bc.shape
    D2 = Wkv.shape[0]
    if out is None:
        out = torch.empty(M, D2, device=Bc.device, dtype=torch.float32)
    check(lib().ltm_project_kv_r(ptr(Bc), ptr(Wkv), ptr(bkv), ptr(out), M, e, D2, PRECISION[precision],
                                 GEMM_IMPL["tcgen05"], stream_ptr(Bc.device)), "project_kv_r")
    return out


def cont_attn_rect_tc(q, KV, X, W, W_out, c_none, jb=None, tb=None, want_scores=False, want_hist=True, n_heads=12):
    """Tensor-core path (num_basis 64/128/256): q[Bv,Q,D], KV[Bv,N,2D] (tf32-rounded) -> (ctx, scores|None, hist|None)."""
    require_cuda(q, KV, X, W, jb, tb)
    q = _f32c(q)
    Bv, Q, D = q.shape
    N = KV.shape[1]
    H, d = n_heads, D // n_heads
    ctx = torch.empty(Bv, Q, D, device=q.device, dtype=torch.float32)
    scores = torch.empty(Bv, H, Q, N, device=q.device, dtype=torch.float32) if want_scores else None
    hist = (torch.empty(Bv, H * ((Q + 31) // 32), STICKY_EDGES - 2, device=q.device, dtype=torch.float32)
            if want_hist else None)
    kv = KV.reshape(Bv * N, 2 * D)
    if attn_tc_split_supported(N, d):          # num_basis 512: two basis halves + combine, histogram from the scores
        if scores is None and want_hist:
            scores = torch.empty(Bv, H, Q, N, device=q.device, dtype=torch.float32)
        part = torch.empty(int(lib().ltm_attn_tc_split_workspace_floats(Bv, Q, H)), device=q.device,
                           dtype=torch.float32)
        check(lib().ltm_cont_attn_rect_tc_split(ptr(q), ptr(kv), C.c_void_p(kv.data_ptr() + 4 * D), 2 * D, ptr(X),
                                                ptr(W), float(W_out), ptr(jb), ptr(tb), ptr(ctx), ptr(scores),
                                                ptr(part), ptr(hist), Bv, Q, N, H, d, stream_ptr(q.device)),
              "cont_attn_rect_tc_split")
        return ctx, (scores if want_scores else None), hist
    check(lib().ltm_cont_attn_rect_tc(ptr(q), ptr(kv), C.c_void_p(kv.data_ptr() + 4 * D), 2 * D, ptr(X), ptr(W),
                                      float(W_out), float(c_none), ptr(jb), ptr(tb), ptr(ctx), ptr(scores), ptr(hist),
                                      Bv, Q, N, H, d, stream_ptr(q.device)), "cont_attn_rect_tc")
    return ctx, scores, hist


def cont_attn_rect_tc16(q, KV16, X16, W, W_out, c_none, jb=None, tb=None, want_scores=False, want_hist=True,
                        n_heads=12):
    """fp16 flavour of `cont_attn_rect_tc`: KV16[Bv,N,2D] float16, X16[N,64] float16 -> (ctx, scores|None, hist|None)."""
    require_cuda(q, KV16, X16, W, jb, tb)
    q = _f32c(q)
    if KV16.dtype != torch.float16 or X16.dtype != torch.float16 or not KV16.is_contiguous():
        raise ValueError("cont_attn_rect_tc16 takes contiguous float16 K|V and X16")
    Bv, Q, D = q.shape
    N = KV16.shape[1]
    H, d = n_heads, D // n_heads
    ctx = torch.empty(Bv, Q, D, device=q.device, dtype=torch.float32)
    scores = torch.empty(Bv, H, Q, N, device=q.device, dtype=torch.float32) if want_scores else None
    hist = (torch.empty(Bv, H * ((Q + 31) // 32), STICKY_EDGES - 2, device=q.device, dtype=torch.float32)
            if want_hist else None)
    kp, vp = C.c_void_p(KV16.data_ptr()), C.c_void_p(KV16.data_ptr() + 2 * D)
    if attn_tc_split_supported(N, d):
        if scores is None and want_hist:
            scores = torch.empty(Bv, H, Q, N, device=q.device, dtype=torch.float32)
        part = torch.empty(int(lib().ltm_attn_tc_split_workspace_floats(Bv, Q, H)), device=q.device,
                           dtype=torch.float32)
        check(lib().ltm_cont_attn_rect_tc16_split(ptr(q), kp, vp, 2 * D, ptr(X16), ptr(W), float(W_out), ptr(jb),
                                                  ptr(tb), ptr(ctx), ptr(scores), ptr(part), ptr(hist), Bv, Q, N, H, d,
                                                  stream_ptr(q.device)), "cont_attn_rect_tc16_split")
        return ctx, (scores if want_scores else None), hist
    check(lib().ltm_cont_attn_rect_tc16(ptr(q), kp, vp, 2 * D, ptr(X16), ptr(W), float(W_out), float(c_none), ptr(jb),
                                        ptr(tb), ptr(ctx), ptr(scores), ptr(hist), Bv, Q, N, H, d,
                                        stream_ptr(q.device)), "cont_attn_rect_tc16")
    return ctx, scores, hist


def project_kv_t(Bcoef, Wkv, bkv, N, precision="tf32", impl="tcgen05", precision_v=None, w_split=None):
    """Same projection with the keys stored transposed per head: -> (Kt[Bv,H,64,N], V[Bv,N,D]).
    `precision_v` (None = `precision`): a different precision for the value half -- the Gaussian variant needs
    fp32-grade keys (softmax(20 S) amplifies score errors 20x) but its values only enter the final contraction."""
    require_cuda(Bcoef, Wkv, bkv)
    Bc = _f32c(Bcoef).reshape(-1, Bcoef.shape[-1])
    M, e = Bc.shape
    D = Wkv.shape[0] // 2
    Bv = M // N
    Kt = torch.empty(Bv, D // 64, 64, N, device=Bc.device, dtype=torch.float32)
    V = torch.empty(Bv, N, D, device=Bc.device, dtype=torch.float32)
    if precision == "fp16x2":
        # both halves as ONE plain fp16 GEMM over K' = 3e on hi/lo-split operands (split_half3): fp32-grade products
        # at the fp16 tensor rate.  W3: the weights split once by the caller ([2D, 3e], side 1).
        A3 = split_half3(Bc, 0)
        W3 = w_split if w_split is not None else split_half3(Wkv, 1)
        g = GemmArgs()
        g.A, g.lda, g.a_kmajor = A3.data_ptr(), 3 * e, 1
        g.B, g.ldb, g.b_kmajor = W3.data_ptr(), 3 * e, 1
        g.K1, g.bias = 3 * e, bkv.data_ptr()
        g.C, g.ldc = V.data_ptr(), D
        g.CT, g.ct_cols, g.ct_group = Kt.data_ptr(), D, N
        g.M, g.Nc, g.K, g.batch = M, 2 * D, 3 * e, 1
        g.precision, g.impl, g.ab_fp16 = PRECISION["tf32"], GEMM_IMPL[impl], 1
        check(lib().ltm_gemm(C.byref(g), stream_ptr(Bc.device)), "project_kv_t(fp16x2)")
        return Kt, V
    if precision_v is not None and (precision_v == "fp16" or PRECISION[precision_v] != PRECISION[precision]):
        g = GemmArgs()                                   # keys: all D columns through the transposed store
        g.A, g.lda, g.a_kmajor = Bc.data_ptr(), e, 1
        g.B, g.ldb, g.b_kmajor = Wkv.data_ptr(), e, 1
        g.K1, g.bias = e, bkv.data_ptr()
        g.C, g.ldc = V.data_ptr(), D                     # (no column takes the row-major path)
        g.CT, g.ct_cols, g.ct_group = Kt.data_ptr(), D, N
        g.M, g.Nc, g.K, g.batch = M, D, e, 1
        g.precision, g.impl = PRECISION[precision], GEMM_IMPL[impl]
        check(lib().ltm_gemm(C.byref(g), stream_ptr(Bc.device)), "project_k_t")
        if precision_v == "fp16":
            # values through kind::f16 UMMAs: coefficients and weights ROUNDED to fp16 first (unbiased; the tensor
            # core would truncate fp32 operands read as tf32, a systematic shrink of V)
            gemm_raw(to_half(Bc), e, 0, True, to_half(Wkv[D:].contiguous()), e, 0, True, V, D, 0, M, D, e, 1,
                     bias=bkv, bias_offset=D, ab_fp16=True, precision="tf32")
        else:
            gemm_raw(Bc, e, 0, True, Wkv, e, 0, True, V, D, 0, M, D, e, 1, bias=bkv, precision=precision_v, impl=impl,
                     b_offset=D * e, bias_offset=D)
        return Kt, V
    check(lib().ltm_project_kv_t(ptr(Bc), ptr(Wkv), ptr(bkv), ptr(Kt), ptr(V), M, e, D, N, PRECISION[precision],
                                 GEMM_IMPL[impl], stream_ptr(Bc.device)), "project_kv_t")
    return Kt, V


def cont_attn_rect_t(q, Kt, V, W, W_out, jb=None, tb=None, want_scores=False, want_hist=True):
    """Fast path (num_basis 64/128/256): q[Bv,Q,D], Kt[Bv,H,64,N], V[Bv,N,D] -> (ctx, scores|None, hist_part|None)."""
    require_cuda(q, Kt, V, W, jb, tb)
    q = _f32c(q)
    Bv, Q, D = q.shape
    H, d, N = Kt.shape[1], Kt.shape[2], Kt.shape[3]
    ctx = torch.empty(Bv, Q, D, device=q.device, dtype=torch.float32)
    scores = torch.empty(Bv, H, Q, N, device=q.device, dtype=torch.float32) if want_scores else None
    hist = (torch.empty(Bv, H * ((Q + 31) // 32), STICKY_EDGES - 2, device=q.device, dtype=torch.float32)
            if want_hist else None)
    check(lib().ltm_cont_attn_rect_t(ptr(q), ptr(Kt), ptr(V), V.stride(1), ptr(W), float(W_out), ptr(jb), ptr(tb),
                                     ptr(ctx), ptr(scores), ptr(hist), Bv, Q, N, H, d, stream_ptr(q.device)),
          "cont_attn_rect_t")
    return ctx, scores, hist


def cont_attn_gauss_t(q, Kt, V, basis_mu, basis_sigma, want_scores=False):
    """Fast path of the Gaussian closed form -> (ctx, scores|None, mu[Bv,H*Q], sd[Bv,H*Q])."""
    require_cuda(q, Kt, V, basis_mu, basis_sigma)
    q = _f32c(q)
    Bv, Q, D = q.shape
    H, d, N = Kt.shape[1], Kt.shape[2], Kt.shape[3]
    ctx = torch.empty(Bv, Q, D, device=q.device, dtype=torch.float32)
    scores = torch.empty(Bv, H, Q, N, device=q.device, dtype=torch.float32) if want_scores else None
    mu = torch.empty(Bv, H * Q, device=q.device, dtype=torch.float32)
    sd = torch.empty(Bv, H * Q, device=q.device, dtype=torch.float32)
    check(lib().ltm_cont_attn_gauss_t(ptr(q), ptr(Kt), ptr(V), V.stride(1), ptr(basis_mu), ptr(basis_sigma), ptr(ctx),
                                      ptr(scores), ptr(mu), ptr(sd), Bv, Q, N, H, d, stream_ptr(q.device)),
          "cont_attn_gauss_t")
    return ctx, scores, mu, sd


def cont_attn_gauss_tc16(q, KV_hi, KV_lo, basis_mu, basis_sigma, n_heads=12):
    """Tensor-core Gaussian closed form: q[Bv,Q,D], KV_hi / KV_lo fp16 [Bv,N,2D] (two-term K|V from the projection
    GEMM) -> (ctx, mu[Bv,H*Q], sd[Bv,H*Q])."""
    require_cuda(q, KV_hi, KV_lo, basis_mu, basis_sigma)
    q = _f32c(q)
    Bv, Q, D = q.shape
    N = KV_hi.shape[1]
    if KV_hi.dtype != torch.float16 or KV_lo.dtype != torch.float16 or KV_hi.shape != KV_lo.shape \
            or not KV_hi.is_contiguous() or not KV_lo.is_contiguous() or KV_hi.shape[2] != 2 * D:
        raise ValueError("cont_attn_gauss_tc16: KV_hi / KV_lo must be contiguous float16 [Bv,N,2D]")
    H = n_heads
    ctx = torch.empty(Bv, Q, D, device=q.device, dtype=torch.float32)
    mu = torch.empty(Bv, H * Q, device=q.device, dtype=torch.float32)
    sd = torch.empty(Bv, H * Q, device=q.device, dtype=torch.float32)
    check(lib().ltm_cont_attn_gauss_tc16(ptr(q), ptr(KV_hi), ptr(KV_lo), 2 * D, ptr(basis_mu), ptr(basis_sigma),
                                         ptr(ctx), ptr(mu), ptr(sd), Bv, Q, N, H, D // H, stream_ptr(q.device)),
          "cont_attn_gauss_tc16")
    return ctx, mu, sd


def project_kv_split(Bcoef, bkv, N, w_split):
    """K|V = B W^T + b as two fp16 terms (hi, lo), [Bv,N,2D] each: one fp16 GEMM over the hi/lo-split operands
    (split_half3) whose epilogue writes the result and its fp16 residual.  w_split: split_half3(Wkv, 1)."""
    require_cuda(Bcoef, bkv, w_split)
    Bc = _f32c(Bcoef).reshape(-1, Bcoef.shape[-1])
    M, e = Bc.shape
    D2 = w_split.shape[0]
    A3 = split_half3(Bc, 0)
    hi = torch.empty(M // N, N, D2, device=Bc.device, dtype=torch.float16)
    lo = torch.empty_like(hi)
    gemm_raw(A3, 3 * e, 0, True, w_split, 3 * e, 0, True, hi, D2, 0, M, D2, 3 * e, 1, bias=bkv, ab_fp16=True,
             c_fp16=True, C_lo=lo, precision="tf32")
    return hi, lo


def cont_attn_rect(q, KV, W, W_out, jb=None, tb=None, n_heads=12, want_scores=False, want_hist=True):
    """q[Bv,Q,D], KV[Bv,N,2D] -> (ctx[Bv,Q,D], scores|None, hist_part|None).  gibbs:224-286."""
    require_cuda(q, KV, W, jb, tb)
    q, KV = _f32c(q), _f32c(KV)
    Bv, Q, D = q.shape
    N = KV.shape[1]
    H = n_heads
    d = D // H
    ctx = torch.empty(Bv, Q, D, device=q.device, dtype=torch.float32)
    scores = torch.empty(Bv, H, Q, N, device=q.device, dtype=torch.float32) if want_scores else None
    hist = (torch.empty(Bv, H * ((Q + 31) // 32), STICKY_EDGES - 2, device=q.device, dtype=torch.float32)
            if want_hist else None)
    check(lib().ltm_cont_attn_rect(ptr(q), ptr(KV), ptr(W), float(W_out), ptr(jb), ptr(tb), ptr(ctx), ptr(scores),
                                   ptr(hist), Bv, Q, N, H, d, stream_ptr(q.device)), "cont_attn_rect")
    return ctx, scores, hist


def cont_attn_gauss(q, KV, basis_mu, basis_sigma, n_heads=12, want_scores=False):
    """-> (ctx[Bv,Q,D], scores|None, mu[Bv,H*Q], sd[Bv,H*Q]).  long_term_attention.py:286-325."""
    require_cuda(q, KV, basis_mu, basis_sigma)
    q, KV = _f32c(q), _f32c(KV)
    Bv, Q, D = q.shape
    N = KV.shape[1]
    H = n_heads
    d = D // H
    ctx = torch.empty(Bv, Q, D, device=q.device, dtype=torch.float32)
    scores = torch.empty(Bv, H, Q, N, device=q.device, dtype=torch.float32) if want_scores else None
    mu = torch.empty(Bv, H * Q, device=q.device, dtype=torch.float32)
    sd = torch.empty(Bv, H * Q, device=q.device, dtype=torch.float32)
    check(lib().ltm_cont_attn_gauss(ptr(q), ptr(KV), ptr(basis_mu), ptr(basis_sigma), ptr(ctx), ptr(scores), ptr(mu),
                                    ptr(sd), Bv, Q, N, H, d, stream_ptr(q.device)), "cont_attn_gauss")
    return ctx, scores, mu, sd


def rbf_eval(tvals, basis_mu, basis_sigma, tidx=None, out=None):
    """out[p,j] = N(t_p; mu_j, sigma_j^2), t_p = tvals[tidx[p]] if tidx is given.  basis_functions.py:158-164."""
    require_cuda(tvals, basis_mu, basis_sigma, tidx)
    P = tidx.numel() if tidx is not None else tvals.numel()
    N = basis_mu.numel()
    if out is None:
        out = torch.empty(P, N, device=tvals.device, dtype=torch.float32)
    check(lib().ltm_rbf_eval(ptr(tvals), ptr(tidx), ptr(basis_mu), ptr(basis_sigma), ptr(out), out.stride(0), P, N,
                             stream_ptr(tvals.device)), "rbf_eval")
    return out


def ridge_solve(positions, trim, rows, basis_mu, basis_sigma, ridge=0.5, want_G=True, want_GT=True):
    """Ridge operator of the Gaussian design, fp64 solve on device.  -> (G[rows,N]|None, GT[N,rows]|None)."""
    require_cuda(positions, basis_mu, basis_sigma)
    P, N = positions.numel(), basis_mu.numel()
    dev = positions.device
    ws = torch.empty(int(lib().ltm_ridge_workspace_doubles(P, N)), device=dev, dtype=torch.float64)
    G = torch.empty(rows, N, device=dev, dtype=torch.float32) if want_G else None
    ld = (rows + 3) // 4 * 4                      # TMA wants 16-byte row pitches
    GTp = torch.zeros(N, ld, device=dev, dtype=torch.float32) if want_GT else None
    check(lib().ltm_ridge_solve(ptr(positions), P, trim, rows, ptr(basis_mu), ptr(basis_sigma), N, float(ridge),
                                ptr(G), ptr(GTp), ld, ptr(ws), stream_ptr(dev)), "ridge_solve")
    return G, (GTp[:, :rows] if want_GT else None)


def gather_rows(src, idx, out=None):
    """out[v,s,:] = src[v, idx[v,s], :]."""
    require_cuda(src, idx)
    Bv, R, e = src.shape
    S = idx.shape[1]
    if out is None:
        out = torch.empty(Bv, S, e, device=src.device, dtype=torch.float32)
    check(lib().ltm_gather_rows(ptr(src), ptr(idx), ptr(out), Bv, R, S, e, stream_ptr(src.device)), "gather_rows")
    return out


def split_half3(x, side):
    """fp32 [rows, K] -> fp16 [rows, 3K]: x ~ hi + lo laid out [hi | lo | hi] (side 0, A operand) or [hi | hi | lo]
    (side 1, B operand), so that a plain fp16 GEMM over 3K gives the three-term split product."""
    require_cuda(x)
    x = _f32c(x)
    rows, K = x.shape
    out = torch.empty(rows, 3 * K, device=x.device, dtype=torch.float16)
    check(lib().ltm_split_half3(ptr(x), ptr(out), rows, K, int(side), stream_ptr(x.device)), "split_half3")
    return out


def fold_sample_columns(GT, b_sorted, S, L, nbins=128):
    """Variant G: per-video update operator with the S sample columns of GT[N, >= S+L] folded per sticky bin
    (b_sorted[Bv,S] ascending) and the L frame columns copied: [Bv, N, nbins + L]."""
    require_cuda(GT, b_sorted)
    if GT.dim() != 2 or GT.stride(1) != 1 or GT.shape[1] < S + L or b_sorted.dtype != torch.int32:
        raise ValueError("fold_sample_columns: GT must be [N, >= S+L] row-major, b_sorted int32 [Bv,S]")
    b_sorted = b_sorted.contiguous()
    Bv, N = b_sorted.shape[0], GT.shape[0]
    out = torch.empty(Bv, N, nbins + L, device=GT.device, dtype=torch.float32)
    check(lib().ltm_fold_sample_columns(ptr(GT), GT.stride(0), ptr(b_sorted), ptr(out), Bv, N, S, L, nbins,
                                        stream_ptr(GT.device)), "fold_sample_columns")
    return out


def _device_guarded(fn):
    """Make the device of the first CUDA tensor argument current for the call (stream handles of one device are
    invalid while another device is current)."""
    import functools

    @functools.wraps(fn)
    def wrapped(*a, **kw):
        for t in list(a) + list(kw.values()):
            if isinstance(t, torch.Tensor) and t.is_cuda:
                if t.device.index != torch.cuda.current_device():
                    with torch.cuda.device(t.device):
                        return fn(*a, **kw)
                break
        return fn(*a, **kw)
    return wrapped


for _name, _fn in list(globals().items()):
    if callable(_fn) and getattr(_fn, "__module__", None) == __name__ and not _name.startswith("_") \
            and not _name.endswith("_supported") and isinstance(_fn, type(_device_guarded)):
        globals()[_name] = _device_guarded(_fn)

