"""Ragged batches through the caller's cross-attention branch (`CrossAttentionLTM.forward(..., lengths=...)`): per-video
chunk lengths on the fp16 tensor-core path, against the lock-step branch bit for bit, against one oracle per video, with
NaN padding, and the three kernels it adds (ragged pool + fp16 convert, GEMM with per-batch extents, softmax with
per-video lengths) on their own."""
import copy

import numpy as np
import pytest
import torch

from oracle import ltm_oracle as O
from tests.helpers import TOL_CTX, compare_draws, relerr

pytestmark = pytest.mark.gpu

TIE = 1e-3


@pytest.fixture(scope="module")
def dev(cuda_device):
    return cuda_device


def _linears(seed, e, D):
    torch.manual_seed(seed)
    return torch.nn.Linear(D, D), torch.nn.Linear(e, D), torch.nn.Linear(e, D)


def _module(dev, lins, alpha=.5, H=12, T=32, N=64, **kw):
    from infinite_video_b200.cross_attention import CrossAttentionLTM
    lq, lk, lv = (copy.deepcopy(x).to(dev) for x in lins)
    return CrossAttentionLTM(lq, lk, lv, alpha, N, .75, n_heads=H, tokens_per_frame=T, **kw)


def _oracle(lins, alpha, T, N=64):
    lq, lk, lv = lins
    return O.CrossAttentionLTM(N, .75, alpha, lq.weight.detach(), lq.bias.detach(), lk.weight.detach(),
                               lk.bias.detach(), lv.weight.detach(), lv.bias.detach(), tokens_per_frame=T,
                               rebuild_tables=False)


def _fresh_pool():
    from infinite_video_b200 import LongTermAttention
    LongTermAttention._shared_pool.update(key=None, x=None, k16=None)


# ------------------------------------------------------------------------------------------------------------------
# 1. equal lengths == lock-step, bit for bit
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape", [
    # e, D, H, Q, T, L, B, videos_per_pass, alpha
    (768, 768, 12, 32, 32, 16, 3, 32, .5),
    (768, 768, 12, 32, 32, 16, 3, 32, 1.0),
    (768, 768, 12, 32, 32, 256, 3, 2, .5),          # Video-LLaMA, two passes (the second holds one video)
    (1024, 768, 12, 96, 196, 4, 2, 32, .5),         # VideoChat2 widths, 784 tokens (not a multiple of 64)
], ids=["vl_small", "vl_alpha1", "vl_two_passes", "vc2_4_frames"])
@pytest.mark.parametrize("masked", [False, True], ids=["nomask", "mask"])
def test_equal_lengths_equal_lockstep(dev, shape, masked):
    """With a general additive mask (normal values x 3, a block at finfo.min) the scale-and-mask step of the softmax
    must round like the lock-step kernel's single FFMA for the bits to agree."""
    e, D, H, Q, T, L, B, vpp, alpha = shape
    lins = _linears(201, e, D)
    a = _module(dev, lins, alpha=alpha, H=H, T=T, videos_per_pass=vpp)
    b = _module(dev, lins, alpha=alpha, H=H, T=T, videos_per_pass=vpp)
    g = torch.Generator().manual_seed(202)
    for c in range(3):
        hidden = torch.randn(B, Q, D, generator=g).to(dev)
        enc = torch.randn(B, L * T, e, generator=g).to(dev)
        u = torch.rand(B, 512, dtype=torch.float64, generator=g)
        mask = None
        if masked:
            mask = torch.randn(B, 1, 1, L * T, generator=g) * 3
            mask[0, ..., : L * T // 3] = torch.finfo(torch.float32).min
            mask = mask.to(dev)
        _fresh_pool()
        ya = a(hidden, enc, new_video=(c == 0), layer=0, u=u, encoder_attention_mask=mask)
        _fresh_pool()
        yb = b(hidden, enc, new_video=(c == 0), layer=0, u=u, lengths=[L] * B, encoder_attention_mask=mask)
        assert torch.equal(ya, yb), c


# ------------------------------------------------------------------------------------------------------------------
# 2. mixed lengths against one oracle per video
# ------------------------------------------------------------------------------------------------------------------
RAGGED = {
    # e, D, H, Q, T, Lmax, plan of lengths per chunk, new_video flags per chunk (None: c == 0)
    "videollama": (768, 768, 12, 32, 32, 16,
                   [[16, 15, 7, 3], [15, 0, 16, 2], [5, 9, 0, 16], [16, 3, 11, 0]],
                   [None, None, [False, False, False, True], None]),
    "videochat2": (1024, 768, 12, 96, 196, 15,
                   [[15, 14, 3], [2, 0, 15], [15, 5, 7]],
                   [None, None, [True, False, False]]),
}


@pytest.mark.parametrize("case", list(RAGGED))
def test_mixed_lengths_match_oracle(dev, case):
    e, D, H, Q, T, Lmax, plan, flags = RAGGED[case]
    B = len(plan[0])
    lins = _linears(211, e, D)
    m = _module(dev, lins, alpha=.5, H=H, T=T)
    orcs = {}
    g = torch.Generator().manual_seed(212)
    worst = 0.0
    for c, lens in enumerate(plan):
        nv = [c == 0] * B if flags[c] is None else flags[c]
        hidden = torch.randn(B, Q, D, generator=g)
        enc = torch.randn(B, Lmax * T, e, generator=g)
        for v, Lv in enumerate(lens):
            enc[v, Lv * T:] = float("nan")
        u = torch.rand(B, 512, dtype=torch.float64, generator=g)
        eng = m.long_term_attention._engine
        before = eng.B_past.clone() if eng is not None and eng.has_state else None
        got = m(hidden.to(dev), enc.to(dev), new_video=torch.tensor(nv), layer=0, u=u, lengths=lens).cpu()
        assert torch.isfinite(got).all(), c
        eng = m.long_term_attention._engine
        for v, Lv in enumerate(lens):
            if Lv == 0:
                assert not got[v].any(), (c, v)
                if before is not None:
                    assert torch.equal(eng.B_past[v], before[v]), (c, v)        # memory carries on untouched
                continue
            if nv[v]:
                orcs[v] = _oracle(lins, .5, T)
            upd = not nv[v]
            b_got = eng.last["b"][v:v + 1].cpu().long() if upd else None
            want = orcs[v].forward(hidden[v:v + 1], enc[v:v + 1, :Lv * T], nv[v], u[v:v + 1] if upd else None,
                                   b_override=b_got)
            if upd:
                compare_draws(b_got, orcs[v].ltm.last["b_own"], u[v:v + 1], orcs[v].ltm.last["p"], TIE)
            err = relerr(got[v:v + 1], want)
            worst = max(worst, err)
            assert err < TOL_CTX, (c, v, Lv, err)
    print(f"\n{case}: worst relerr vs the per-video oracle {worst:.2e}")


# ------------------------------------------------------------------------------------------------------------------
# 3. the padding is never read
# ------------------------------------------------------------------------------------------------------------------
def test_padding_never_read(dev):
    e, D, H, Q, T, L, B = 768, 768, 12, 32, 32, 12, 4
    lins = _linears(221, e, D)
    a = _module(dev, lins)
    b = _module(dev, lins)
    g = torch.Generator().manual_seed(222)
    for c, lens in enumerate([[12, 5, 0, 2], [3, 12, 7, 0], [0, 9, 12, 2]]):
        hidden = torch.randn(B, Q, D, generator=g).to(dev)
        enc = torch.randn(B, L * T, e, generator=g)
        mask = torch.where(torch.rand(B, 1, 1, L * T, generator=g) < .3, -1e4, 0.0)
        encn, maskn = enc.clone(), mask.clone()
        for v, Lv in enumerate(lens):
            enc[v, Lv * T:] = 0.0
            encn[v, Lv * T:] = float("nan")
            maskn[v, ..., Lv * T:] = float("nan")
        u = torch.rand(B, 512, dtype=torch.float64, generator=g)
        nv = torch.tensor([[True] * 4, [False, False, True, False], [False] * 4][c])   # slot 2 refilled at chunk 1
        ya = a(hidden, enc.to(dev), new_video=nv, u=u, encoder_attention_mask=mask.to(dev), lengths=lens)
        yb = b(hidden, encn.to(dev), new_video=nv, u=u, encoder_attention_mask=maskn.to(dev), lengths=lens)
        assert torch.isfinite(yb).all() and torch.equal(ya, yb), c


# ------------------------------------------------------------------------------------------------------------------
# 4. the kernels on their own
# ------------------------------------------------------------------------------------------------------------------
def _offs(lens, dev):
    return torch.tensor(np.concatenate([[0], np.cumsum(lens)]), dtype=torch.int32, device=dev)


@pytest.mark.parametrize("T,e,lens", [(32, 768, [5, 0, 8, 2]), (196, 1024, [15, 3, 0]), (7, 64, [3, 9, 2])])
def test_pool_mean_convert_ragged(dev, T, e, lens):
    from infinite_video_b200 import ops
    g = torch.Generator().manual_seed(T)
    B, L = len(lens), max(lens)
    k = torch.randn(B, L, T, e, generator=g).to(dev)
    for v, Lv in enumerate(lens):
        k[v, Lv:] = float("nan")
    ld16 = (L * T + 63) // 64 * 64
    frames = sum(lens)
    for splits in (1, 3):
        x, k16 = ops.pool_mean_convert_ragged(k, _offs(lens, dev), frames, splits, ld16 + 64)
        assert k16.shape == (B, ld16 + 64, e)
        want = torch.empty(frames, splits, e, device=dev)
        from infinite_video_b200._capi import check, lib, ptr, stream_ptr
        check(lib().ltm_pool_mean_ragged(ptr(k), 0, ptr(want), ptr(_offs(lens, dev)), B, L, T, e, splits, frames, 0,
                                         stream_ptr(dev)), "pool_mean_ragged")
        assert torch.equal(x, want), splits
    # sentinel past roundup64(n_v): untouched
    sentinel = torch.full((B, ld16 + 64, e), 7.0, device=dev, dtype=torch.float16)
    from infinite_video_b200._capi import check, lib, ptr, stream_ptr
    xp = torch.empty(frames, 1, e, device=dev)
    check(lib().ltm_pool_mean_convert_ragged(ptr(k), ptr(xp), ptr(sentinel), ptr(_offs(lens, dev)), B, L, T, e, 1,
                                             frames, ld16 + 64, stream_ptr(dev)), "pool_mean_convert_ragged")
    for v, Lv in enumerate(lens):
        n = Lv * T
        n64 = (n + 63) // 64 * 64
        tok = k[v, :Lv].reshape(n, e)
        if n:
            assert torch.equal(sentinel[v, :n].view(torch.int16), ops.to_half(tok).view(torch.int16)), v
        tail = sentinel[v, n:n64]
        assert torch.equal(tail.view(torch.int16), torch.zeros_like(tail).view(torch.int16)), v      # +0.0
        assert (sentinel[v, n64:] == 7.0).all(), v


def _gemm_ref(A, B, b_kmajor, n_v, k_v):
    """fp64 product of batch b over its first k_v K-elements: A[M, K] x B (K-major [N, K] or MN-major [K, N])."""
    Bm = B.double() if not b_kmajor else B.double().transpose(0, 1)
    return A[:, :k_v].double() @ Bm[:k_v]


@pytest.mark.parametrize("b_kmajor", [True, False], ids=["kmajor", "mnmajor"])
@pytest.mark.parametrize("M,N", [(384, 2936), (96, 400)])
def test_gemm_extents(dev, b_kmajor, M, N):
    from infinite_video_b200 import ops
    g = torch.Generator().manual_seed(M + N)
    K = 3008 if not b_kmajor else 1024                      # MN-major: the values GEMM (K = tokens)
    batch = 4
    A = (torch.randn(batch, M, K, generator=g) * .1).half().to(dev)
    Bt = (torch.randn(batch, N, K, generator=g) * .1).half() if b_kmajor else \
        (torch.randn(batch, K, N, generator=g) * .1).half()
    Bt = Bt.to(dev)
    ldb = K if b_kmajor else N
    Kb = [0, 64, K // 2 // 64 * 64, K] if not b_kmajor else [K] * batch
    nb = [N, 0, 131, N] if b_kmajor else [N] * batch
    C_ = torch.full((batch, M, N), 12345.0, device=dev)
    ne = torch.tensor(nb, dtype=torch.int32, device=dev)
    ke = torch.tensor(Kb, dtype=torch.int32, device=dev)
    ops.gemm_raw(A, K, M * K, True, Bt, ldb, Bt.shape[1] * Bt.shape[2], b_kmajor, C_, N, M * N, M, N, K, batch,
                 precision="tf32", ab_fp16=True, n_ext=ne if b_kmajor else None, k_ext=None if b_kmajor else ke)
    C_ = C_.cpu()
    for b in range(batch):
        want = _gemm_ref(A[b].cpu(), Bt[b].cpu(), b_kmajor, nb[b], Kb[b])
        if nb[b] == 0 or Kb[b] == 0:
            assert (C_[b] == 12345.0).all(), b                 # an empty batch leaves C unwritten
            continue
        bn = 256 if (N > 128 and -(-N // 256) * -(-M // 128) * batch >= 74) else 128
        ncols = min(N, -(-nb[b] // bn) * bn)                  # whole tiles up to the one holding column n_ext - 1
        assert relerr(C_[b, :, :ncols], want[:, :ncols]) < 1e-4, b
        assert (C_[b, :, ncols:] == 12345.0).all(), b        # tiles past the extent are skipped
    # full extents: the bits of ltm_gemm
    full = torch.empty(batch, M, N, device=dev)
    ref = torch.empty(batch, M, N, device=dev)
    ops.gemm_raw(A, K, M * K, True, Bt, ldb, Bt.shape[1] * Bt.shape[2], b_kmajor, full, N, M * N, M, N, K, batch,
                 precision="tf32", ab_fp16=True, n_ext=torch.full((batch,), N, dtype=torch.int32, device=dev),
                 k_ext=torch.full((batch,), (K + 63) // 64 * 64, dtype=torch.int32, device=dev))
    ops.gemm_raw(A, K, M * K, True, Bt, ldb, Bt.shape[1] * Bt.shape[2], b_kmajor, ref, N, M * N, M, N, K, batch,
                 precision="tf32", ab_fp16=True)
    assert torch.equal(full, ref)


def _fp16_ulp(p):
    ex = torch.floor(torch.log2(p.abs().clamp_min(2.0 ** -14)))
    return torch.pow(2.0, ex - 10)


@pytest.mark.parametrize("ld,n_v,rpl", [(3008, [2940, 0, 1, 2999, 64], 8), (12352, [12301, 8192, 0], 4)])
def test_softmax_rows_h_len(dev, ld, n_v, rpl):
    from infinite_video_b200 import ops
    g = torch.Generator().manual_seed(ld)
    V = len(n_v)
    S = torch.randn(V * rpl, ld, generator=g) * 50
    mask = torch.where(torch.rand(V, ld + 4, generator=g) < .4, -1e4, 0.0)
    for v, n in enumerate(n_v):
        S[v * rpl:(v + 1) * rpl, n:] = float("nan")
        mask[v, n:] = float("nan")
    mask = mask.contiguous()
    nl = torch.tensor(n_v, dtype=torch.int32, device=dev)
    Sd = S.to(dev)
    for m in (None, mask):
        P = torch.full((V * rpl, ld), 3.0, dtype=torch.float16, device=dev)
        from infinite_video_b200._capi import check, lib, ptr, stream_ptr
        md = None if m is None else m.to(dev)
        check(lib().ltm_softmax_rows_h_len(ptr(Sd), ptr(md), ptr(P), ptr(nl), V * rpl, ld,
                                           0 if m is None else m.shape[1], rpl, .125, stream_ptr(dev)), "softmax_len")
        P = P.cpu()
        for v, n in enumerate(n_v):
            rows = slice(v * rpl, (v + 1) * rpl)
            n64 = (n + 63) // 64 * 64
            if n == 0:
                assert (P[rows] == 3.0).all()
                continue
            logits = S[rows, :n].double() * .125 + (0 if m is None else m[v, :n].double())
            want = torch.softmax(logits, -1)
            ulps = ((P[rows, :n].double() - want).abs() / _fp16_ulp(want)).max()
            assert float(ulps) <= 1.0, (v, float(ulps))
            assert not P[rows, n:n64].any() and not torch.signbit(P[rows, n:n64].float()).any()
            assert (P[rows, n64:] == 3.0).all()
    # the wrapper returns the same probabilities
    Pw = ops.softmax_rows_half_len(S.to(dev).nan_to_num(), nl, rpl, .125).cpu()
    for v, n in enumerate(n_v):
        if n:
            assert torch.isfinite(Pw[v * rpl:(v + 1) * rpl, :n]).all()


# ------------------------------------------------------------------------------------------------------------------
# 5. errors before any launch
# ------------------------------------------------------------------------------------------------------------------
def test_errors_before_any_launch(dev, monkeypatch):
    from infinite_video_b200 import ops
    from infinite_video_b200.batched import BatchedRectLTM
    e, Q, L, T, B = 768, 8, 4, 32, 3
    lins = _linears(231, e, e)
    m = _module(dev, lins)
    hidden = torch.randn(B, Q, e, device=dev)
    enc = torch.randn(B, L * T, e, device=dev)
    m(hidden, enc, new_video=True, lengths=[4, 0, 2])               # slot 1 holds no memory now
    gauss = _module(dev, lins, variant="gaussian")
    fp32 = _module(dev, lins, operands="fp32")
    launched = []
    for name in ("gemm_raw", "to_half", "softmax_rows", "softmax_rows_half", "softmax_rows_half_len", "blend",
                 "pool_mean_convert_ragged", "pool_mean"):
        monkeypatch.setattr(ops, name, lambda *a, _n=name, **kw: launched.append(_n))
    monkeypatch.setattr(BatchedRectLTM, "pool", lambda *a, **kw: launched.append("pool"))
    monkeypatch.setattr(BatchedRectLTM, "step", lambda *a, **kw: launched.append("step"))
    cases = [(m, dict(lengths=[4, 1, 2], new_video=True)),           # a one-frame chunk
             (m, dict(lengths=[4, 5, 2], new_video=True)),           # longer than the chunk
             (m, dict(lengths=[4, 2], new_video=True)),              # one length short
             (m, dict(lengths=[4, 2.5, 2], new_video=True)),         # not an integer
             (m, dict(lengths=torch.tensor([4, 2, 2], device=dev), new_video=True)),
             (m, dict(lengths=[4, 2, 2], new_video=False)),          # slot 1 has no memory
             (m, dict(lengths=[4, 2, 2], new_video=torch.tensor([False, False, True], device=dev))),
             (fp32, dict(lengths=[4, 2, 2], new_video=True)),
             (gauss, dict(lengths=[4, 2, 2], new_video=True))]
    for mod, kw in cases:
        with pytest.raises(ValueError):
            mod(hidden, enc, **kw)
    with pytest.raises(ValueError):                                   # 40 queries inside videos that had 8
        m(torch.randn(B, 40, e, device=dev), enc, new_video=False, lengths=[4, 0, 2])
    with pytest.raises(NotImplementedError):
        gauss(hidden, enc, lengths=[4, 2, 2], new_video=True)
    with pytest.raises(ValueError):
        m.short_term(hidden, enc, lengths=[4, 1, 2])
    with pytest.raises(ValueError):
        fp32.short_term(hidden, enc, lengths=[4, 2, 2])
    assert launched == [], launched
    assert gauss.long_term_attention._engine is None and fp32.long_term_attention._engine is None


def test_pool_with_half_ragged_and_alpha_one(dev):
    """BatchedRectLTM.pool(with_half=True, lengths=) returns the packed frames and the padded fp16 chunk; 16-bit chunks
    with with_half still raise.  alpha == 1 with lengths is the ragged short-term context alone."""
    from infinite_video_b200.batched import BatchedRectLTM
    e, L, T, B = 768, 7, 32, 3
    lins = _linears(241, e, e)
    eng = BatchedRectLTM(64, .75, lins[1].weight.detach(), lins[1].bias.detach(), lins[2].weight.detach(),
                         lins[2].bias.detach(), device=dev)
    k = torch.randn(B, L * T, e, device=dev)
    lens = [7, 0, 3]
    x, k16 = eng.pool(k, with_half=True, lengths=lens)
    assert torch.equal(x, eng.pool(k, lengths=lens)) and k16.shape == (B, 256, e)
    with pytest.raises(ValueError):
        eng.pool(k.half(), with_half=True, lengths=lens)
    m = _module(dev, lins, alpha=1.0)
    hidden = torch.randn(B, 32, e, device=dev)
    got = m(hidden, k, lengths=lens)
    assert m.long_term_attention._engine is None and not got[1].any()
    q = m._linear(hidden.reshape(B * 32, e), m.query, "tf32x3").view(B, 32, e)
    for v, Lv in enumerate(lens):
        if Lv:
            want = m.short_term(q[v:v + 1], k[v:v + 1, :Lv * T].contiguous())
            assert relerr(got[v:v + 1], want) < TOL_CTX, v


def test_all_videos_idle(dev):
    """A batch in which every video is idle: zero rows, no error, and every video's memory carried on to its next
    chunk, which then matches a module that never saw the idle call."""
    e, Q, L, T, B = 768, 32, 6, 32, 3
    lins = _linears(251, e, e)
    for alpha in (.5, 1.0):
        a, b = _module(dev, lins, alpha=alpha), _module(dev, lins, alpha=alpha)
        g = torch.Generator().manual_seed(252)
        hidden = [torch.randn(B, Q, e, generator=g).to(dev) for _ in range(2)]
        enc = [torch.randn(B, L * T, e, generator=g).to(dev) for _ in range(3)]
        u = torch.rand(B, 512, dtype=torch.float64, generator=g)
        lens = [6, 4, 2]
        a(hidden[0], enc[0], new_video=True, lengths=lens)
        b(hidden[0], enc[0], new_video=True, lengths=lens)
        idle = a(hidden[1], enc[1], new_video=False, u=u, lengths=[0] * B)
        assert not idle.any(), alpha
        _fresh_pool()
        ya = a(hidden[1], enc[2], new_video=False, u=u, lengths=lens)
        _fresh_pool()
        yb = b(hidden[1], enc[2], new_video=False, u=u, lengths=lens)
        assert torch.equal(ya, yb), alpha
