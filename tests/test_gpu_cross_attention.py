"""The caller's cross-attention branch (`CrossAttentionLTM`, INTEGRATION.md section 4) against a plain float64
reference: short-term attention at the Video-LLaMA and VideoChat2 widths, over several passes, with HF encoder masks in
both value conventions, with 16-bit inputs, and the small kernels of stm.cu (row softmax, blend, fp16 copy) at their
edges.  Each short-term case prints its measured error."""
import copy
import math

import pytest
import torch

from oracle import ltm_oracle as O
from tests.helpers import TOL_CTX, relerr

pytestmark = pytest.mark.gpu

FMIN = torch.finfo(torch.float32).min
MASKED = {"m10000": -10000.0, "finfo_min": FMIN}          # the two values HF has used for a masked token
PATTERNS = ("none", "last40", "every_third_frame", "one_frame_left", "all")


@pytest.fixture(scope="module")
def dev(cuda_device):
    return cuda_device


def _ops():
    from infinite_video_b200 import ops
    return ops


def _linears(seed, e, D):
    torch.manual_seed(seed)
    return torch.nn.Linear(D, D), torch.nn.Linear(e, D), torch.nn.Linear(e, D)


def _module(dev, lins, alpha=.5, H=12, T=32, **kw):
    from infinite_video_b200.cross_attention import CrossAttentionLTM
    lq, lk, lv = (copy.deepcopy(x).to(dev) for x in lins)
    return CrossAttentionLTM(lq, lk, lv, alpha, 64, .75, n_heads=H, tokens_per_frame=T, **kw)


def stm_fp64(q, enc, lk, lv, H, mask=None):
    """softmax(q_h K_h^T / sqrt(d) + mask) V_h in float64 on q's device, with K = enc Wk^T + bk and V = enc Wv^T + bv
    formed as the reference module forms them (no re-association).  q[B,Q,D], enc[B,LT,e], mask additive [B,1,1,LT]."""
    dv = q.device
    q, enc = q.double(), enc.to(dv).double()
    wk, bk, wv, bv = (t.detach().to(dv).double() for t in (lk.weight, lk.bias, lv.weight, lv.bias))
    B, Q, D = q.shape
    LT, d = enc.shape[1], D // H
    K = (enc @ wk.T + bk).view(B, LT, H, d).transpose(1, 2)
    V = (enc @ wv.T + bv).view(B, LT, H, d).transpose(1, 2)
    s = q.view(B, Q, H, d).transpose(1, 2) @ K.transpose(-1, -2) / math.sqrt(d)
    if mask is not None:
        s = s + mask.to(dv).double().reshape(B, 1, 1, LT)
    return (torch.softmax(s, -1) @ V).transpose(1, 2).reshape(B, Q, D)


def _masked_tokens(kind, L, T):
    """bool [L*T]: the tokens one video masks."""
    m = torch.zeros(L, T, dtype=torch.bool)
    if kind == "last40":
        m.view(-1)[int(round(.6 * L * T)):] = True
    elif kind == "every_third_frame":
        m[::3] = True
    elif kind == "one_frame_left":
        m[:] = True
        m[L // 2] = False
    elif kind == "all":
        m[:] = True
    else:
        assert kind == "none"
    return m.view(-1)


def _hf_mask(kinds, L, T, value):
    """HF's extended encoder mask [B,1,1,LT]: 0 for kept tokens, `value` for masked ones, one pattern per video."""
    m = torch.stack([_masked_tokens(k, L, T) for k in kinds])
    return torch.where(m, torch.tensor(value), torch.tensor(0.0)).view(len(kinds), 1, 1, L * T)


def _count_softmax(monkeypatch, ops):
    calls = {"fp32": 0, "fp16": 0}

    def wrap(fn, key):
        def counted(*a, **kw):
            calls[key] += 1
            return fn(*a, **kw)
        return counted
    monkeypatch.setattr(ops, "softmax_rows", wrap(ops.softmax_rows, "fp32"))
    monkeypatch.setattr(ops, "softmax_rows_half", wrap(ops.softmax_rows_half, "fp16"))
    return calls


# ------------------------------------------------------------------------------------------------------------------
# (a) the float64 reference
# ------------------------------------------------------------------------------------------------------------------
def test_reference_matches_the_oracle(dev):
    """The float64 reference against the oracle's fp32 short-term context (`last_stm`, bit-identical to the real
    `BertSelfAttention`), at the VideoChat2 widths with a mask in both conventions and a fully masked video."""
    lq, lk, lv = _linears(41, 1024, 768)
    B, Q, L, T = 4, 16, 2, 196
    g = torch.Generator().manual_seed(42)
    hidden = torch.randn(B, Q, 768, generator=g)
    enc = torch.randn(B, L * T, 1024, generator=g)
    orc = O.CrossAttentionLTM(64, .75, 1.0, lq.weight.detach(), lq.bias.detach(), lk.weight.detach(),
                              lk.bias.detach(), lv.weight.detach(), lv.bias.detach(), tokens_per_frame=T,
                              rebuild_tables=False)
    q64 = torch.nn.functional.linear(hidden.double(), lq.weight.detach().double(), lq.bias.detach().double())
    kinds = ("none", "last40", "one_frame_left", "all")
    for value in MASKED.values():
        mask = _hf_mask(kinds, L, T, value)
        for v in range(B):
            orc.forward(hidden[v:v + 1], enc[v:v + 1], True, mask=mask[v:v + 1])
            want = stm_fp64(q64[v:v + 1].to(dev), enc[v:v + 1], lk, lv, 12, mask[v:v + 1]).cpu()
            # on a video masked everywhere with -10000 the oracle's fp32 sum `scores - 10000` rounds every score to a
            # multiple of 2^-10, which moves each probability by up to 2^-11 of itself
            tol = 1e-3 if (value == -10000.0 and kinds[v] == "all") else 1e-5
            assert relerr(orc.last_stm, want) < tol, (value, v)


# ------------------------------------------------------------------------------------------------------------------
# (b) short_term against float64
# ------------------------------------------------------------------------------------------------------------------
SHAPES = {
    # name: e, D, H, Q, T, L, B, videos_per_pass
    "videollama_two_passes": (768, 768, 12, 32, 32, 256, 3, 2),     # 8192 tokens; the second pass holds one video
    "videochat2": (1024, 768, 12, 96, 196, 16, 2, 32),              # BASELINE cfg3: 3136 tokens, fp16 operands
    "videochat2_15_frames": (1024, 768, 12, 96, 196, 15, 2, 32),    # 2940 tokens: L*T % 8 != 0 -> the fp32 path
    "h16_e1024": (1024, 1024, 16, 40, 32, 64, 2, 32),               # 2048 tokens
}


@pytest.mark.parametrize("operands", ["fp16", "fp32"])
@pytest.mark.parametrize("shape", list(SHAPES))
def test_short_term_against_fp64(dev, shape, operands, monkeypatch):
    e, D, H, Q, T, L, B, vpp = SHAPES[shape]
    ops = _ops()
    lins = _linears(51, e, D)
    m = _module(dev, lins, H=H, T=T, operands=operands, videos_per_pass=vpp)
    g = torch.Generator().manual_seed(52)
    q = (torch.randn(B, Q, D, generator=g) * 2).to(dev)
    enc = torch.randn(B, L * T, e, generator=g).to(dev)
    calls = _count_softmax(monkeypatch, ops)
    got = m.short_term(q, enc)
    err = relerr(got, stm_fp64(q, enc, lins[1], lins[2], H))
    print(f"\nshort_term {shape} operands={operands}: relerr vs fp64 {err:.2e}")
    half = operands == "fp16" and (L * T) % 8 == 0 and e % 8 == 0
    passes = -(-B // vpp)
    assert calls == ({"fp32": 0, "fp16": passes} if half else {"fp32": passes, "fp16": 0}), calls
    if shape == "videochat2_15_frames":
        assert calls["fp16"] == 0                      # the fp32 fallback inside operands="fp16"
    assert m.long_term_attention._engine is None       # short_term alone never builds the LTM engine
    assert err < TOL_CTX, err


# ------------------------------------------------------------------------------------------------------------------
# (c) encoder masks
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("convention", list(MASKED))
@pytest.mark.parametrize("operands", ["fp16", "fp32"])
def test_short_term_with_masks(dev, operands, convention):
    """One pattern per video.  (i) Every video matches float64 with the same mask; the fully masked video gets uniform
    weights under finfo.min and its unmasked result under -10000.  (ii) Masked probabilities are exactly 0, so a new
    draw of the masked tokens of `enc` leaves every video that keeps a token bit-identical."""
    e, D, H, Q, T, L = 768, 768, 12, 32, 32, 64
    B = len(PATTERNS)
    lins = _linears(61, e, D)
    m = _module(dev, lins, operands=operands)
    g = torch.Generator().manual_seed(62)
    q = (torch.randn(B, Q, D, generator=g) * 2).to(dev)
    enc = torch.randn(B, L * T, e, generator=g)
    mask = _hf_mask(PATTERNS, L, T, MASKED[convention])
    got = m.short_term(q, enc.to(dev), mask.to(dev))
    want = stm_fp64(q, enc, lins[1], lins[2], H, mask)
    errs = [relerr(got[v], want[v]) for v in range(B)]
    print(f"\nmasks operands={operands} {convention}: relerr vs fp64 per video "
          + " ".join(f"{p} {x:.2e}" for p, x in zip(PATTERNS, errs)))
    assert max(errs) < TOL_CTX, errs
    full = PATTERNS.index("all")
    if convention == "finfo_min":          # uniform weights: what zero scores give
        alt = stm_fp64(torch.zeros_like(q[full:full + 1]), enc[full:full + 1], lins[1], lins[2], H)
    else:                                  # -10000 shifts every score alike: the unmasked result
        alt = stm_fp64(q[full:full + 1], enc[full:full + 1], lins[1], lins[2], H)
    assert relerr(got[full], alt[0]) < TOL_CTX
    # (ii)
    masked = mask.view(B, L * T, 1) != 0
    enc2 = torch.where(masked, torch.randn(enc.shape, generator=g) * 3, enc)
    got2 = m.short_term(q, enc2.to(dev), mask.to(dev))
    for v in range(B):
        if v != full:
            assert torch.equal(got2[v], got[v]), (PATTERNS[v], float((got2[v] - got[v]).abs().max()))
    assert not torch.equal(got2[full], got[full])


def test_masks_are_validated_before_any_launch(dev, monkeypatch):
    """forward, short_term and ops.softmax_rows* refuse a mask the kernels would read out of bounds or from the wrong
    video, before anything is launched."""
    ops = _ops()
    B, Q, L, T, e = 2, 8, 4, 32, 768
    lins = _linears(71, e, e)
    m = _module(dev, lins, operands="fp16")
    hidden = torch.randn(B, Q, e, device=dev)
    enc = torch.randn(B, L * T, e, device=dev)
    launched = []
    for name in ("gemm_raw", "to_half", "softmax_rows", "softmax_rows_half", "blend"):
        monkeypatch.setattr(ops, name, lambda *a, _n=name, **kw: launched.append(_n))
    bad = [torch.zeros(1, 1, 1, L * T, device=dev),              # one mask broadcast over two videos
           torch.zeros(B, 1, Q, L * T, device=dev),              # per query
           torch.zeros(B, 12, 1, L * T, device=dev),             # per head
           torch.zeros(B, 1, 1, L * T - 8, device=dev),          # wrong L*T
           torch.zeros(B, 1, 1, L * T, device=dev, dtype=torch.bool),
           torch.zeros(B, 1, 1, L * T)]                          # on the host
    for mask in bad:
        with pytest.raises(ValueError):
            m(hidden, enc, new_video=True, encoder_attention_mask=mask)
        with pytest.raises(ValueError):
            m.short_term(hidden, enc, mask)
    assert launched == [] and m.long_term_attention._engine is None
    monkeypatch.undo()
    ops = _ops()
    n, rpm = 64, 4
    S = torch.randn(2 * rpm, n, device=dev)
    S0 = S.clone()
    good = torch.zeros(2, n, device=dev)
    for mask, r in [(torch.zeros(1, n, device=dev), rpm),               # one row short: the second half reads past it
                    (torch.zeros(3, n, device=dev), rpm),               # one row too many
                    (good, 3),                                          # rows_per_mask does not divide the rows
                    (good, 0),
                    (good.half(), rpm),
                    (torch.zeros(n, 2, device=dev).t(), rpm),           # not contiguous
                    (good.cpu(), rpm),
                    (torch.zeros(2, n // 2, device=dev), rpm)]:         # two rows of half the width
        with pytest.raises(ValueError):
            ops.softmax_rows(S, .5, mask, r)
        with pytest.raises(ValueError):
            ops.softmax_rows_half(S, .5, mask, r)
    torch.cuda.synchronize()
    assert torch.equal(S, S0)
    ops.softmax_rows(S, .5, good, rpm)                                   # and the right one runs
    assert torch.allclose(S.sum(-1), torch.ones(2 * rpm, device=dev))


# ------------------------------------------------------------------------------------------------------------------
# (d) several passes
# ------------------------------------------------------------------------------------------------------------------
def test_passes_give_the_same_bits(dev):
    """forward with 7 videos, a mask and the fp16 chunk copy of the LTM's pooling pass, in 7, 3 or 1 pass(es) of
    videos: every video's rows go through the same per-row K order, whatever the pass (and the GEMM tile width that
    the pass size selects), so the results are identical."""
    from infinite_video_b200 import LongTermAttention
    e, Q, T, L, B = 768, 32, 32, 64, 7
    lins = _linears(81, e, e)
    m = _module(dev, lins, alpha=.5)
    g = torch.Generator().manual_seed(82)
    hidden = torch.randn(B, Q, e, generator=g).to(dev)
    enc = torch.randn(B, L * T, e, generator=g).to(dev)
    mask = _hf_mask([PATTERNS[v % len(PATTERNS)] for v in range(B)], L, T, FMIN).to(dev)
    outs = {}
    for vpp in (1, 3, 32):
        m.videos_per_pass = vpp
        outs[vpp] = m(hidden, enc, new_video=True, layer=0, encoder_attention_mask=mask)
        assert LongTermAttention._shared_pool["k16"] is not None          # the fp16 copy came from the pooling pass
    assert torch.equal(outs[1], outs[3]) and torch.equal(outs[1], outs[32])
    # and that short-term context is the float64 one
    q = m._linear(hidden.reshape(B * Q, e), m.query, "tf32x3").view(B, Q, e)
    for vpp in (1, 3, 32):
        m.videos_per_pass = vpp
        assert relerr(m.short_term(q, enc, mask), stm_fp64(q, enc, lins[1], lins[2], 12, mask)) < TOL_CTX


# ------------------------------------------------------------------------------------------------------------------
# (e) input dtypes and alpha
# ------------------------------------------------------------------------------------------------------------------
def test_fp16_inputs_equal_the_fp32_module(dev):
    """fp16 hidden states, chunk and mask (autocast in VideoChat2): the output is the fp32 module's on the up-cast
    inputs, cast to fp16, bit for bit, over 3 chunks of two modules stepped in lock-step."""
    e, D, Q, T, L, B = 1024, 768, 96, 196, 16, 2
    lins = _linears(91, e, D)
    m16, m32 = _module(dev, lins, T=T), _module(dev, lins, T=T)
    g = torch.Generator().manual_seed(92)
    for c in range(3):
        hidden = torch.randn(B, Q, D, generator=g).to(dev).half()
        enc = torch.randn(B, L * T, e, generator=g).to(dev).half()
        mask = _hf_mask([PATTERNS[(v + c) % 4] for v in range(B)], L, T, -10000.0).to(dev).half()
        u = torch.rand(B, 512, dtype=torch.float64, generator=g)
        got = m16(hidden, enc, new_video=(c == 0), layer=0, encoder_attention_mask=mask, u=u)
        want = m32(hidden.float(), enc.float(), new_video=(c == 0), layer=0, encoder_attention_mask=mask.float(), u=u)
        assert got.dtype == torch.float16 and want.dtype == torch.float32
        assert torch.equal(got, want.half()), c


def test_alpha_one_is_the_short_term_context(dev):
    e, Q, T, L, B = 768, 32, 32, 16, 3
    lins = _linears(101, e, e)
    m = _module(dev, lins, alpha=1.0)
    g = torch.Generator().manual_seed(102)
    hidden = torch.randn(B, Q, e, generator=g).to(dev)
    enc = torch.randn(B, L * T, e, generator=g).to(dev)
    mask = _hf_mask(PATTERNS[1:4], L, T, FMIN).to(dev)
    got = m(hidden, enc, new_video=True, encoder_attention_mask=mask)
    assert m.long_term_attention._engine is None
    q = m._linear(hidden.reshape(B * Q, e), m.query, "tf32x3").view(B, Q, e)
    assert torch.equal(got, m.short_term(q, enc, mask))
    q64 = torch.nn.functional.linear(hidden.double(), lins[0].weight.detach().to(dev).double(),
                                     lins[0].bias.detach().to(dev).double())
    assert relerr(got, stm_fp64(q64, enc, lins[1], lins[2], 12, mask)) < TOL_CTX


# ------------------------------------------------------------------------------------------------------------------
# (f) the kernels of stm.cu at their edges
# ------------------------------------------------------------------------------------------------------------------
def _softmax_case(dev, rows, n, rows_per_mask, value, seed):
    """Scores x 50 (the max subtraction matters) and one mask row per `rows_per_mask` score rows, cycling through
    no mask, the last 40 %, every third token, all but one token, every token and a random half."""
    g = torch.Generator().manual_seed(seed)
    S = torch.randn(rows, n, generator=g) * 50
    nm = rows // rows_per_mask
    masked = torch.zeros(nm, n, dtype=torch.bool)
    for i in range(nm):
        kind = i % 6
        if kind == 1:
            masked[i, int(round(.6 * n)):] = True
        elif kind == 2:
            masked[i, ::3] = True
        elif kind == 3:
            masked[i] = True
            masked[i, n // 2] = False
        elif kind == 4:
            masked[i] = True
        elif kind == 5:
            masked[i] = torch.rand(n, generator=g) < .5
            masked[i, 0] = False
    mask = torch.where(masked, torch.tensor(value), torch.tensor(0.0))
    # the kernel adds the mask to the fp32 logit S * scale (exact for scale = 1/8); the reference is the float64
    # softmax of that fp32 sum.  It differs from the exact one only on a row masked everywhere with -10000, where
    # the fp32 sum rounds the scores to 2^-10 (as PyTorch's fp32 softmax does)
    logits = (S * .125).view(nm, rows_per_mask, n) + mask.view(nm, 1, n)
    want = torch.softmax(logits.double(), -1).view(rows, n)
    return S, mask, masked.repeat_interleave(rows_per_mask, 0), want


@pytest.mark.parametrize("value", list(MASKED.values()), ids=list(MASKED))
@pytest.mark.parametrize("rows_per_mask", [1, 12 * 32])
@pytest.mark.parametrize("n", [4, 1020, 2940, 8192, 12288])
def test_softmax_rows_fp32(dev, n, rows_per_mask, value):
    ops = _ops()
    rows = 6 * rows_per_mask
    S, mask, masked, want = _softmax_case(dev, rows, n, rows_per_mask, value, seed=n + rows_per_mask)
    P = ops.softmax_rows(S.to(dev), .125, mask.to(dev), rows_per_mask).cpu()
    err = float(((P.double() - want).abs().amax(-1) / want.abs().amax(-1)).max())
    assert err < 2e-6, err
    assert float((P.double().sum(-1) - 1).abs().max()) < 1e-5
    partial = masked & ~masked.all(-1, keepdim=True)
    assert not P[partial].any()                 # a masked token of a row that keeps one has probability exactly 0
    # without a mask
    S2 = S[:4].to(dev)
    P2 = ops.softmax_rows(S2, .125).cpu()
    assert relerr(P2, torch.softmax(S[:4].double() * .125, -1)) < 2e-6


def _fp16_ulp(p):
    """Spacing of the fp16 grid at p (float64): 2^(e - 10) for normal magnitudes, 2^-24 in the subnormal range."""
    ex = torch.floor(torch.log2(p.abs().clamp_min(2.0 ** -14)))
    return torch.pow(2.0, ex - 10)


@pytest.mark.parametrize("value", list(MASKED.values()), ids=list(MASKED))
@pytest.mark.parametrize("n,rows_per_mask", [(4, 1), (4, 8), (12, 24), (8196, 8), (12288, 40)])
def test_softmax_rows_half_within_one_fp16_ulp(dev, n, rows_per_mask, value):
    """n <= 8192: the register-resident kernel; above: the three-pass kernel.  Every fp16 probability is within one
    fp16 ulp of the float64 one."""
    ops = _ops()
    rows = 6 * rows_per_mask
    S, mask, masked, want = _softmax_case(dev, rows, n, rows_per_mask, value, seed=7 * n + rows_per_mask)
    P = ops.softmax_rows_half(S.to(dev), .125, mask.to(dev), rows_per_mask).cpu()
    assert P.dtype == torch.float16
    dev_ulps = ((P.double() - want).abs() / _fp16_ulp(want)).max()
    assert float(dev_ulps) <= 1.0, float(dev_ulps)
    partial = masked & ~masked.all(-1, keepdim=True)
    assert not P[partial].any()


BLEND_ROUND = 148 * 8 * 256 * 4          # elements one grid-stride round of the blend kernel covers


@pytest.mark.parametrize("n", [4, 2 * BLEND_ROUND + 12])
def test_blend(dev, n):
    ops = _ops()
    g = torch.Generator().manual_seed(n % 1000)
    a = torch.randn(n, generator=g) * torch.pow(2.0, torch.randint(-20, 20, (n,), generator=g).float())
    b = torch.randn(n, generator=g)
    ad, bd = a.to(dev), b.to(dev)
    assert torch.equal(ops.blend(ad, bd, 1.0).cpu(), a)
    assert torch.equal(ops.blend(ad, bd, 0.0).cpu(), b)
    # the kernel takes alpha as a float and computes 1 - alpha in float: the reference uses the same two weights
    al = float(torch.tensor(0.9, dtype=torch.float32))
    be = float(1 - torch.tensor(al, dtype=torch.float32))
    got = ops.blend(ad, bd, 0.9).cpu().double()
    want = al * a.double() + be * b.double()
    scale = al * a.double().abs() + be * b.double().abs()
    ulp = torch.pow(2.0, torch.floor(torch.log2(scale.clamp_min(2.0 ** -126))) - 23)
    assert float(((got - want).abs() / ulp).max()) <= 2.0


HALF_ROUND = 148 * 16 * 256 * 8          # elements one grid-stride round of the fp16 copy covers


@pytest.mark.parametrize("n", [8, HALF_ROUND + 8 * 37])
def test_to_half_is_round_to_nearest_even(dev, n):
    """Overflow to +-inf (|x| >= 65520), subnormal results, ties, NaN: the copy equals x.half() bit for bit."""
    ops = _ops()
    g = torch.Generator().manual_seed(n % 1000)
    x = torch.randn(n, generator=g) * torch.pow(2.0, torch.randint(-30, 18, (n,), generator=g).float())
    special = torch.tensor([65504.0, 65519.99, 65520.0, -65520.0, 1e6, -3e38, float("inf"), float("-inf"),
                            float("nan"), 2.0 ** -24, 2.0 ** -25, 3 * 2.0 ** -26, -(2.0 ** -25) * 1.0001, 2.0 ** -14,
                            2.0 ** -14 - 2.0 ** -25, 1e-9, -0.0, 1 + 2.0 ** -11, 1 + 3 * 2.0 ** -11, -1e-30])
    k = min(len(special), n)
    x[:k] = special[:k]
    x[-k:] = special[:k].flip(0)
    if n > HALF_ROUND:
        x[HALF_ROUND - k // 2:HALF_ROUND - k // 2 + k] = special[:k]
    got = ops.to_half(x.to(dev)).cpu()
    want = x.half()
    nan = torch.isnan(want)
    assert torch.equal(torch.isnan(got), nan)
    assert torch.equal(got.view(torch.int16)[~nan], want.view(torch.int16)[~nan])
    if n > 8:
        assert torch.isinf(want).any() and (want.abs() < 2.0 ** -14).logical_and(want != 0).any()
