"""N1 (SURVEY section 8f): the cross-attention branch of the Q-former's `BertSelfAttention` -- short-term softmax
attention over the chunk's L*T encoder tokens plus the (1 - alpha) LTM context -- on libinfltm.

Reference: infty-Video-LLaMA/InfVideoLLaMA/models/Qformer.py:197-310
    q = query(hidden)                                   :211
    a_long = LTM(enc, q, new_video)   iff alpha != 1    :216-223
    K, V = key(enc), value(enc)                         :225-226     (two [L*T, e] x [e, 768] GEMMs)
    probs = softmax(q_h K_h^T / sqrt(d) + mask)         :241, :279-285
    ctx = probs V                                       :297-300
    out = alpha * ctx + (1 - alpha) * a_long            :303-304

The short-term half is re-associated so that K and V of the 8192 tokens are never materialised:
    scores_h = (q_h W_k,h) enc^T / sqrt(d)      (+ q_h.b_k,h, a per-row constant: softmax-invariant, dropped)
    ctx_h    = (probs_h enc) W_v,h^T + b_v,h    (rows of probs sum to 1)
which halves the flops (9.7 instead of 19.3+ GFLOP per video-chunk at L*T = 8192) and removes 100 MB of K/V
traffic per video.  Every contraction runs on the tcgen05 GEMM (`ltm_gemm`), the row softmax and the blend are two
small streaming kernels.  The key/value projections are the ones the LTM shares (`proj_key=self.key`, :156-157).
"""
import math

import numpy as np
import torch
import torch.nn as nn

from . import ops
from .batched import _as_lengths
from .ltm import LongTermAttention


class RaggedUnsupported(NotImplementedError, ValueError):
    """Per-video lengths with a configuration that has no ragged path (the Gaussian LTM variant): an unsupported
    feature (NotImplementedError) and an invalid argument combination (ValueError), raised before any launch."""


def encoder_mask_rows(mask, B, LT, device=None):
    """The caller's additive encoder mask as a contiguous float32 [B, LT] (one row per video, shared by every head and
    query), or None.  Accepted: [B, LT], [B, 1, LT] and [B, 1, 1, LT] in any float dtype -- the last is what HF's
    `invert_attention_mask` makes of a 2-D mask over the encoder tokens, in the model's dtype (fp16 under autocast).
    Anything else raises ValueError: a mask of batch 1 broadcast over B > 1 videos, a mask that varies per query or
    per head, a wrong LT, an integer or boolean mask, or (with `device`) a mask on another device."""
    if mask is None:
        return None
    shape = tuple(mask.shape)
    if shape not in ((B, LT), (B, 1, LT), (B, 1, 1, LT)):
        raise ValueError(f"encoder_attention_mask of shape {list(shape)}: expected [B, LT], [B, 1, LT] or "
                         f"[B, 1, 1, LT] with B = {B}, LT = {LT} (per-query and per-head masks are not supported)")
    if not mask.is_floating_point():
        raise ValueError(f"encoder_attention_mask must be an additive float mask, got {mask.dtype}")
    if device is not None and mask.device != torch.device(device):
        raise ValueError(f"encoder_attention_mask is on {mask.device}, the chunk on {device}")
    return mask.reshape(B, LT).float().contiguous()


class CrossAttentionLTM(nn.Module):
    """Drop-in for the cross-attention use of `BertSelfAttention` (eval mode, absolute position embeddings, no head
    mask).  Construct from the caller's own `query` / `key` / `value` `nn.Linear`s and its config values."""

    def __init__(self, query: nn.Linear, key: nn.Linear, value: nn.Linear, alpha: float, num_basis: int, tau: float,
                 sticky: bool = True, n_heads: int = 12, tokens_per_frame: int = 32, videos_per_pass: int = 32,
                 precision: str = "tf32x3", score_precision: str = None, value_precision: str = None,
                 operands: str = "fp16", **ltm_kwargs):
        super().__init__()
        self.query, self.key, self.value = query, key, value
        self.alpha = float(alpha)
        self.H = n_heads
        self.d = query.out_features // n_heads
        # bounds the [videos, H*Q, L*T] score buffer (12.6 MB per video at L*T = 8192); large passes amortise the
        # host side of the five GEMM launches, which is what bounds small batches
        self.videos_per_pass = videos_per_pass
        self.precision = precision
        # the two large contractions (scores = Qt enc^T, Y = probs enc); the three small ones always run split-TF32.
        # Measured (scripts/stm_probe.py, error vs fp64 at L*T = 8192 / 256, time at 16 videos):
        #   scores x1 (Qt rounded to tf32) / values x3   2.6e-4 / 2.1e-4   0.80 ms
        #   scores x3 / values x1                         4.5e-4 / 9.4e-4   0.87 ms
        #   x1 / x1                                       5.8e-4 / 9.2e-4   0.59 ms
        #   x3 / x3                                       3.9e-5 / 1.2e-5   1.08 ms   <- default
        # (a single pass reads the raw chunk, which the tensor core truncates: a bias that shrinks every score by about
        # 2^-11 of itself, so its error grows with the logits.  Single-pass scores reach 1.1e-3 at logits of std 1.2,
        # VideoChat2 widths (tests/test_gpu_cross_attention.py): split-TF32 scores are the default.  This is also the
        # path "fp16" operands fall back to, where it must not be less accurate than the fp16 path it stands in for)
        self.score_precision = score_precision or precision
        self.value_precision = value_precision or "tf32x3"
        # operands of the two large contractions.  "fp16" (default): the chunk tokens are converted ONCE per chunk to
        # fp16 with round-to-nearest (one streaming pass, 25 -> 12.6 MB per video), `Qt` and the probabilities are
        # produced as fp16, and both contractions run as kind::f16 UMMAs (twice the TF32 rate, half the operand bytes;
        # the values need no split: rounding is unbiased where the tensor core's truncation of fp32 was not).
        # "fp32": the TF32 / split-TF32 path described above.
        if operands not in ("fp16", "fp32"):
            raise ValueError("operands must be 'fp16' or 'fp32'")
        self.operands = operands
        self.long_term_attention = LongTermAttention(
            head_size=self.d, length=key.in_features, target_len=key.in_features, attn_func="softmax",
            attn_num_basis=num_basis, continuous=True, attn_drop=0.1, infinite_memory=True, n_layers=2,
            n_heads=n_heads, affines=True, mask=True, mask_type="cnn", kl_regularizer=False, proj_key=key,
            proj_value=value, sigma_0=None, mu_0=None, sticky_memories=sticky, sigmas=None, tau=tau,
            d_model=query.out_features, tokens_per_frame=tokens_per_frame, **ltm_kwargs)

    def _linear(self, x, lin, precision):
        """x[M, in] @ W^T + b on tcgen05."""
        M, K = x.shape
        out = torch.empty(M, lin.out_features, device=x.device, dtype=torch.float32)
        w = lin.weight.detach().float().contiguous()
        b = None if lin.bias is None else lin.bias.detach().float().contiguous()
        return ops.gemm_raw(x, K, 0, True, w, K, 0, True, out, lin.out_features, 0, M, lin.out_features, K, 1,
                            bias=b, precision=precision)

    def _ragged_lengths(self, B, LT, e, lengths):
        """Validated per-video lengths (frames) of a ragged call, before anything is launched."""
        if self.operands != "fp16":
            raise ValueError("per-video lengths need operands='fp16' (the fp32 path reads the padding of the chunk)")
        T = self.long_term_attention.tokens_per_frame
        if e % 8:
            raise ValueError(f"per-video lengths need a token width that is a multiple of 8, got {e}")
        if LT % T or LT // T < 2:
            raise ValueError(f"the chunk has {LT} tokens: a ragged chunk is padded to L*{T} tokens, L >= 2")
        return _as_lengths(lengths, B, LT // T)

    @torch.no_grad()
    def short_term(self, q, enc, mask=None, enc16=None, lengths=None):
        """softmax(q_h K_h^T / sqrt(d) + mask) V_h for all heads.  q[B,Q,D] (already projected), enc[B,LT,e] fp32,
        mask: additive, one row per video ([B, LT], [B, 1, LT] or [B, 1, 1, LT], `encoder_mask_rows`) or None; enc16:
        the chunk as float16 when the caller already has it (the pooling pass of the LTM writes it,
        `LongTermAttention.pool_for_caller`).  Returns [B,Q,D].
        lengths: per-video chunk lengths in frames (host ints, 0 = idle, else in [2, L]); video v attends over its
        first n_v = lengths[v] * T tokens only -- the rest of its chunk and of its mask row is never read -- and the
        rows of idle videos are zero.  enc16 is then the padded fp16 chunk [B, ld16, e] of `pool_for_caller(enc,
        lengths)` (ld16 = L*T rounded up to 64 tokens)."""
        B, Q, D = q.shape
        LT, e = enc.shape[1], enc.shape[2]
        H, d = self.H, self.d
        dev = q.device
        if lengths is not None:
            lens = self._ragged_lengths(B, LT, e, lengths)
            mask = encoder_mask_rows(mask, B, LT, dev)
            return self._short_term_ragged(q, enc, mask, enc16, lens)
        mask = encoder_mask_rows(mask, B, LT, dev)
        wk = self.key.weight.detach().float().contiguous()          # [D, e]
        wv = self.value.weight.detach().float().contiguous()
        bv = self.value.bias.detach().float().contiguous() if self.value.bias is not None else None
        out = torch.empty(B, Q, D, device=dev, dtype=torch.float32)
        for v0 in range(0, B, self.videos_per_pass):
            nb = min(self.videos_per_pass, B - v0)
            qv = q[v0:v0 + nb].contiguous()
            ev = enc[v0:v0 + nb].contiguous()
            if self.operands == "fp16" and e % 8 == 0 and LT % 8 == 0:
                # [nb, LT, e] fp16, rounded: from the LTM's pooling pass, or converted here
                e16 = enc16[v0:v0 + nb].contiguous() if enc16 is not None else ops.to_half(ev)
                # (1) Qt as fp16, straight out of the (split-TF32) GEMM epilogue
                Qt = torch.empty(nb, H, Q, e, device=dev, dtype=torch.float16)
                ops.gemm_raw(qv, D, d, True, wk, e, d * e, False, Qt, e, Q * e, nb * Q, e, d, H,
                             c_group=Q, c_group_stride=H * Q * e, precision="tf32x3", c_fp16=True)
                # (2) scores[v] = Qt[v] enc[v]^T : both operands fp16, K-major
                S = torch.empty(nb, H * Q, LT, device=dev, dtype=torch.float32)
                ops.gemm_raw(Qt, e, H * Q * e, True, e16, e, LT * e, True, S, LT, H * Q * LT, H * Q, LT, e, nb,
                             precision="tf32", ab_fp16=True)
                # (3) probabilities as fp16
                m = None if mask is None else mask[v0:v0 + nb]
                P = ops.softmax_rows_half(S, 1.0 / math.sqrt(d), m, H * Q)
                # (4) Yh[h][v][q][:] = probs enc[v] : A fp16 K-major, B = enc16[v] read as [K = LT][N = e] (MN-major)
                Yh = torch.empty(H, nb, Q, e, device=dev, dtype=torch.float32)
                ops.gemm_raw(P, LT, H * Q * LT, True, e16, e, LT * e, False, Yh, e, Q * e, H * Q, e, LT, nb,
                             c_group=Q, c_group_stride=nb * Q * e, precision="tf32", ab_fp16=True)
                # (5) as below
                ops.gemm_raw(Yh, e, nb * Q * e, True, wv, e, d * e, True, out, D, d, nb * Q, d, e, H,
                             bias=bv, bias_stride=d, precision="tf32x3", c_offset=v0 * Q * D)
                continue
            # (1) Qt[v][h][q][:] = q_h W_k,h : batch over heads, A = column block h of q, B = row block h of W_k
            #     read as [K = d][N = e] (MN-major); rows m = (v, q) land at (v*H + h)*Q + q
            Qt = torch.empty(nb, H, Q, e, device=dev, dtype=torch.float32)
            ops.gemm_raw(qv, D, d, True, wk, e, d * e, False, Qt, e, Q * e, nb * Q, e, d, H,
                         c_group=Q, c_group_stride=H * Q * e, precision="tf32x3",
                         round_tf32=(self.score_precision == "tf32"))   # rounded (not truncated) operand of (2)
            # (2) scores[v] = Qt[v] enc[v]^T : [H*Q, e] x [e, LT]
            S = torch.empty(nb, H * Q, LT, device=dev, dtype=torch.float32)
            ops.gemm_raw(Qt, e, H * Q * e, True, ev, e, LT * e, True, S, LT, H * Q * LT, H * Q, LT, e, nb,
                         precision=self.score_precision)
            # (3) probs = softmax(scores / sqrt(d) + mask), in place
            m = None if mask is None else mask[v0:v0 + nb]
            ops.softmax_rows(S, 1.0 / math.sqrt(d), m, H * Q)
            # (4) Yh[h][v][q][:] = probs[v][(h,q)] enc[v] : B operand = enc[v] read as [K = LT][N = e] (MN-major)
            Yh = torch.empty(H, nb, Q, e, device=dev, dtype=torch.float32)
            ops.gemm_raw(S, LT, H * Q * LT, True, ev, e, LT * e, False, Yh, e, Q * e, H * Q, e, LT, nb,
                         c_group=Q, c_group_stride=nb * Q * e, precision=self.value_precision)
            # (5) ctx[:, h*d:(h+1)*d] = Yh[h] W_v,h^T + b_v,h : batch over heads
            ops.gemm_raw(Yh, e, nb * Q * e, True, wv, e, d * e, True, out, D, d, nb * Q, d, e, H,
                         bias=bv, bias_stride=d, precision="tf32x3", c_offset=v0 * Q * D)
        return out

    def _short_term_ragged(self, q, enc, mask, enc16, lens):
        """The short-term half of a ragged batch on the fp16 path.  Per video v, n_v = lengths[v] * T tokens:
        scores through the GEMM with column extents n_v (S rows of pitch ld16), the softmax over the first n_v columns
        with a zero tail up to roundup64(n_v), the values GEMM over roundup64(n_v) tokens (k16 and P hold zeros past
        n_v), then the per-head GEMM as in the lock-step path.  Idle videos get no tiles and zero rows."""
        B, Q, D = q.shape
        LT, e = enc.shape[1], enc.shape[2]
        H, d = self.H, self.d
        T = self.long_term_attention.tokens_per_frame
        dev = q.device
        ld16 = (LT + 63) // 64 * 64
        n = np.asarray(lens, np.int64) * T
        idle = np.flatnonzero(n == 0)
        # one upload: n_v [B] | roundup64(n_v) [B] | frame offsets [B+1] | idle videos
        host = np.concatenate([n, (n + 63) // 64 * 64, np.concatenate([[0], np.cumsum(lens)]), idle]).astype(np.int32)
        ext = torch.from_numpy(host).pin_memory().to(dev, non_blocking=True)
        n_dev, k_dev, offs = ext[:B], ext[B:2 * B], ext[2 * B:3 * B + 1]
        if enc16 is None:
            L = LT // T
            enc16 = ops.pool_mean_convert_ragged(enc.contiguous().view(B, L, T, e), offs, int(sum(lens)), 1, ld16)[1]
        elif enc16.dtype != torch.float16 or tuple(enc16.shape) != (B, ld16, e) or not enc16.is_contiguous():
            raise ValueError(f"enc16 of a ragged call must be a contiguous float16 [{B}, {ld16}, {e}] tensor")
        wk = self.key.weight.detach().float().contiguous()          # [D, e]
        wv = self.value.weight.detach().float().contiguous()
        bv = self.value.bias.detach().float().contiguous() if self.value.bias is not None else None
        out = torch.empty(B, Q, D, device=dev, dtype=torch.float32)
        for v0 in range(0, B, self.videos_per_pass):
            nb = min(self.videos_per_pass, B - v0)
            if not any(lens[v0:v0 + nb]):
                continue                                 # every video of the pass idle: rows zeroed below
            qv = q[v0:v0 + nb].contiguous()
            e16 = enc16[v0:v0 + nb]
            ne, ke = n_dev[v0:v0 + nb], k_dev[v0:v0 + nb]
            Qt = torch.empty(nb, H, Q, e, device=dev, dtype=torch.float16)
            ops.gemm_raw(qv, D, d, True, wk, e, d * e, False, Qt, e, Q * e, nb * Q, e, d, H,
                         c_group=Q, c_group_stride=H * Q * e, precision="tf32x3", c_fp16=True)
            # scores: tiles of video v with a first column >= n_v are skipped
            S = torch.empty(nb, H * Q, ld16, device=dev, dtype=torch.float32)
            ops.gemm_raw(Qt, e, H * Q * e, True, e16, e, ld16 * e, True, S, ld16, H * Q * ld16, H * Q, LT, e, nb,
                         precision="tf32", ab_fp16=True, n_ext=ne)
            m = None if mask is None else mask[v0:v0 + nb]
            P = ops.softmax_rows_half_len(S, ne, H * Q, 1.0 / math.sqrt(d), m)
            # values over the first roundup64(n_v) tokens of video v (P and k16 are zero past n_v)
            Yh = torch.empty(H, nb, Q, e, device=dev, dtype=torch.float32)
            ops.gemm_raw(P, ld16, H * Q * ld16, True, e16, e, ld16 * e, False, Yh, e, Q * e, H * Q, e, ld16, nb,
                         c_group=Q, c_group_stride=nb * Q * e, precision="tf32", ab_fp16=True, k_ext=ke)
            ops.gemm_raw(Yh, e, nb * Q * e, True, wv, e, d * e, True, out, D, d, nb * Q, d, e, H,
                         bias=bv, bias_stride=d, precision="tf32x3", c_offset=v0 * Q * D)
        if len(idle):
            # (Yh of an idle video is never written: its rows of `out` are garbage until here)
            out.index_fill_(0, ext[3 * B + 1:].long(), 0.0)
        return out

    @torch.no_grad()
    def forward(self, hidden_states, encoder_hidden_states, new_video=False, layer=None,
                encoder_attention_mask=None, u=None, lengths=None):
        """Returns the blended context layer [B,Q,D] (what `BertSelfAttention.forward` returns as outputs[0]).
        lengths: per-video chunk lengths in frames of a ragged batch (host ints, 0 = idle, else in [2, L]; the
        chunk is padded to L frames and its padding is never read).  new_video is then a bool or one host flag per
        video; idle videos keep their memory and get zero rows.  Needs operands='fp16' and the 'gibbs' LTM variant."""
        if not hidden_states.is_cuda:
            raise RuntimeError("CrossAttentionLTM runs on CUDA tensors only (no CPU fallback)")
        B, Q, _ = hidden_states.shape
        # HF additive mask [B,1,1,LT] -> [B,LT], validated before anything is launched
        enc = encoder_hidden_states
        mask = encoder_mask_rows(encoder_attention_mask, B, enc.shape[1], enc.device)
        ltm = self.long_term_attention
        if lengths is not None:
            lens = self._ragged_lengths(B, enc.shape[1], enc.shape[2], lengths)
            if self.alpha != 1.0:
                if ltm.variant != "gibbs":
                    raise RaggedUnsupported("per-video lengths exist for the 'gibbs' LTM variant only")
                ltm.check_ragged(enc, lens, new_video, Q)
            enc = enc.float().contiguous()
            q = self._linear(hidden_states.float().reshape(B * Q, -1).contiguous(), self.query, "tf32x3").view(B, Q, -1)
            enc16 = ltm.pool_for_caller(enc, lens) if (self.alpha != 1.0 and ltm.share_pooling) else None
            ctx = self._short_term_ragged(q, enc, mask, enc16, lens)
            if self.alpha == 1.0:
                return ctx.to(hidden_states.dtype)
            a_long = ltm(enc, q, new_doc=new_video, layer_n=layer, u=u, lengths=lens)
            return ops.blend(ctx, a_long.float(), self.alpha).to(hidden_states.dtype)
        enc = enc.float().contiguous()
        q = self._linear(hidden_states.float().reshape(B * Q, -1).contiguous(), self.query, "tf32x3")
        q = q.view(B, Q, -1)
        enc16 = None
        if (self.alpha != 1.0 and self.operands == "fp16" and ltm.variant == "gibbs" and ltm.share_pooling
                and enc.dtype == torch.float32 and enc.is_contiguous() and enc.shape[2] % 8 == 0 and enc.shape[1] % 8 == 0
                and enc.shape[1] % ltm.tokens_per_frame == 0):
            # one pass over the chunk: pooled frames for the LTM (parked in its shared-pooling slot) + the fp16 copy
            # the short-term GEMMs read
            enc16 = ltm.pool_for_caller(enc)
        ctx = self.short_term(q, enc, mask, enc16=enc16)
        if self.alpha == 1.0:
            return ctx.to(hidden_states.dtype)
        a_long = self.long_term_attention(enc, q, new_doc=new_video, layer_n=layer, u=u)
        return ops.blend(ctx, a_long.float(), self.alpha).to(hidden_states.dtype)
