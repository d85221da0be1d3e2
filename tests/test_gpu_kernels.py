"""Per-kernel parity: every libinfltm entry point (through the C-ABI / ctypes) against the CPU oracle on the
same seeded inputs.  Integer / index outputs bit-exact; floating point within the stated tolerance."""
import math

import numpy as np
import pytest
import torch

from oracle import ltm_oracle as O
from tests.helpers import make_inputs, make_proj, proj_tensors, relerr

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev(cuda_device):
    return cuda_device


def _ops():
    from infinite_video_b200 import ops
    return ops


def _tables():
    from infinite_video_b200 import tables
    return tables


# ---------------------------------------------------------------------------------------- R4
@pytest.mark.parametrize("Bv,L,T,e,splits", [(2, 8, 32, 768, 1), (2, 8, 32, 768, 4), (1, 16, 196, 1024, 1),
                                             (1, 16, 196, 1024, 7), (3, 5, 9, 772, 2)])
def test_pool_mean(dev, Bv, L, T, e, splits):
    g = torch.Generator().manual_seed(1)
    k = torch.randn(Bv, L, T, e, generator=g)
    want = k.mean(dim=2)                                    # gibbs:304
    got = _ops().pool_mean(k.to(dev), splits).sum(2).cpu()
    assert relerr(got, want) < 1e-6


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
@pytest.mark.parametrize("Bv,L,T,e,splits", [(2, 8, 32, 768, 1), (1, 16, 196, 1024, 5)])
def test_pool_mean_16bit_inputs(dev, dtype, Bv, L, T, e, splits):
    """fp16 / bf16 chunks (VideoChat2 fp16 autocast) are pooled from their storage with fp32 accumulation."""
    g = torch.Generator().manual_seed(2)
    k = torch.randn(Bv, L, T, e, generator=g).to(dtype)
    want = k.float().mean(dim=2)
    got = _ops().pool_mean(k.to(dev), splits).sum(2).cpu()
    assert relerr(got, want) < 1e-6


@pytest.mark.parametrize("Bv,L,T,e,splits", [(2, 8, 32, 768, 1), (2, 8, 32, 768, 4), (1, 16, 196, 1024, 7),
                                             (3, 5, 9, 776, 2)])
def test_pool_mean_convert(dev, Bv, L, T, e, splits):
    """One pass: pooled partial sums bit-identical to `pool_mean`, fp16 copy identical to a round-to-nearest cast."""
    g = torch.Generator().manual_seed(3)
    k = (torch.randn(Bv, L, T, e, generator=g) * 3).to(dev)
    x, k16 = _ops().pool_mean_convert(k, splits)
    assert torch.equal(x, _ops().pool_mean(k, splits))
    assert torch.equal(k16, k.half())


@pytest.mark.parametrize("Bv,N,L,T,e", [(3, 256, 256, 32, 768), (2, 512, 256, 32, 768), (2, 64, 16, 196, 1024),
                                        (2, 64, 8, 32, 768), (1, 100, 64, 9, 772), (2, 128, 256, 4, 768)])
def test_pool_bins(dev, Bv, N, L, T, e):
    """Per-bin pooling == summing the per-frame pooling over the frames of each bin, in frame order, bit for bit."""
    ops, tb = _ops(), _tables()
    t = tb.rect_tables(L, N, 0.75, 512)
    g = torch.Generator().manual_seed(4)
    k = (torch.randn(Bv, L, T, e, generator=g) * 2).to(dev)
    got = ops.pool_bins(k, t.to(dev)["fbin_ptr"], t.xb_rows)
    x = ops.pool_mean(k, 1)[:, :, 0]                                   # [Bv, L, e]
    want = torch.zeros_like(got)
    for r in range(t.xb_rows):
        for f in range(int(t.fbin_ptr[r]), int(t.fbin_ptr[r + 1])):
            want[:, r] += x[:, f]
    assert torch.equal(got, want)


def test_split_half3_gives_fp32_grade_products_on_fp16_tensor_cores(dev):
    """x ~ hi + lo in fp16, laid out [hi|lo|hi] x [hi|hi|lo] along K: a plain fp16 GEMM over 3K is the three-term split
    product -- as accurate as split-TF32 (4e-6 vs 6e-6 here), far beyond a single fp16 / tf32 pass (5e-4)."""
    ops = _ops()
    g = torch.Generator().manual_seed(13)
    M, Nc, K = 384, 256, 768
    A = (torch.randn(M, K, generator=g) * 3).to(dev)
    W = (torch.randn(Nc, K, generator=g) / 28).to(dev)
    bias = torch.randn(Nc, generator=g).to(dev)
    A3, W3 = ops.split_half3(A, 0), ops.split_half3(W, 1)
    hi = A.half()
    assert torch.equal(A3[:, :K], hi) and torch.equal(A3[:, 2 * K:], hi) and torch.equal(W3[:, K:2 * K], W.half())
    assert torch.equal(A3[:, K:2 * K], (A - hi.float()).half())
    out = torch.zeros(M, Nc, device=dev)
    ops.gemm_raw(A3, 3 * K, 0, True, W3, 3 * K, 0, True, out, Nc, 0, M, Nc, 3 * K, 1, bias=bias, ab_fp16=True,
                 precision="tf32")
    want = A.double() @ W.double().t() + bias.double()
    x3 = torch.zeros(M, Nc, device=dev)
    ops.gemm_raw(A, K, 0, True, W, K, 0, True, x3, Nc, 0, M, Nc, K, 1, bias=bias, precision="tf32x3")
    e16, e32 = relerr(out, want), relerr(x3, want)
    assert e16 < 1e-5 and e16 < 2 * e32, (e16, e32)


@pytest.mark.parametrize("ctas", [1, 5, 64])
def test_gemm_with_a_bounded_grid_is_bit_identical(dev, ctas):
    """ltm_gemm_args.max_ctas: the persistent kernel walks the same tiles with fewer CTAs -- same bits."""
    ops = _ops()
    g = torch.Generator().manual_seed(15)
    M, Nc, K = 1500, 700, 320
    A = torch.randn(M, K, generator=g).to(dev)
    W = torch.randn(Nc, K, generator=g).to(dev)
    bias = torch.randn(Nc, generator=g).to(dev)
    full = torch.zeros(M, Nc, device=dev)
    few = torch.zeros(M, Nc, device=dev)
    for prec in ("tf32", "tf32x3"):
        ops.gemm_raw(A, K, 0, True, W, K, 0, True, full, Nc, 0, M, Nc, K, 1, bias=bias, precision=prec)
        ops.gemm_raw(A, K, 0, True, W, K, 0, True, few, Nc, 0, M, Nc, K, 1, bias=bias, precision=prec, max_ctas=ctas)
        assert torch.equal(full, few), prec


def test_gemm_two_term_fp16_output(dev):
    """ltm_gemm c_fp16 + C_lo: the result as two fp16 terms, hi + lo within 2^-21 of the fp32 result."""
    ops = _ops()
    g = torch.Generator().manual_seed(14)
    M, Nc, K = 300, 192, 256
    A = torch.randn(M, K, generator=g).to(dev)
    W = torch.randn(Nc, K, generator=g).to(dev)
    bias = torch.randn(Nc, generator=g).to(dev)
    hi = torch.zeros(M, Nc, device=dev, dtype=torch.float16)
    lo = torch.zeros_like(hi)
    ops.gemm_raw(A, K, 0, True, W, K, 0, True, hi, Nc, 0, M, Nc, K, 1, bias=bias, precision="tf32x3", c_fp16=True, C_lo=lo)
    full = torch.zeros(M, Nc, device=dev)
    ops.gemm_raw(A, K, 0, True, W, K, 0, True, full, Nc, 0, M, Nc, K, 1, bias=bias, precision="tf32x3")
    assert torch.equal(hi, full.half())
    assert torch.equal(lo, (full - hi.float()).half())
    assert relerr(hi.float() + lo.float(), full) < 5e-7


@pytest.mark.parametrize("N,Bv,Q", [(256, 3, 32), (64, 2, 32), (128, 2, 40), (256, 1, 96)])
def test_cont_attn_gauss_on_tensor_cores(dev, N, Bv, Q):
    """Tensor-core Gaussian attention (two-term fp16 operands, csrc/attn_g16.cu) against the fp32 FMA kernel on the same
    keys / values, and both against an fp64 evaluation: the density parameters and the context."""
    ops, T = _ops(), _tables()
    g = torch.Generator().manual_seed(N + Q)
    H, d, D = 12, 64, 768
    t = T.gauss_tables(8, N, .75)
    bmu, bsig = torch.from_numpy(t.basis_mu).to(dev), torch.from_numpy(t.basis_sigma).to(dev)
    q = torch.randn(Bv, Q, D, generator=g).to(dev)
    KV = (torch.randn(Bv, N, 2 * D, generator=g) * 0.5).to(dev)
    KV[:, :, D:] *= 3.0
    hi = KV.half()
    lo = (KV - hi.float()).half()
    ctx, mu, sd = ops.cont_attn_gauss_tc16(q, hi, lo, bmu, bsig)
    Kt = KV[:, :, :D].reshape(Bv, N, H, d).permute(0, 2, 3, 1).contiguous()
    V = KV[:, :, D:].contiguous()
    ctx_f, _, mu_f, sd_f = ops.cont_attn_gauss_t(q, Kt, V, bmu, bsig)
    # fp64 reference
    K64 = KV[:, :, :D].double().view(Bv, N, H, d).transpose(1, 2)
    V64 = KV[:, :, D:].double().view(Bv, N, H, d).transpose(1, 2)
    qh = q.double().view(Bv, Q, H, d).transpose(1, 2) / 8.0
    a = torch.softmax(20 * (qh @ K64.transpose(-1, -2)), -1)
    bm, bs = bmu.double(), bsig.double()
    m = a @ bm
    var = a @ (bm ** 2 + bs ** 2) - m ** 2
    s = torch.sqrt(bs ** 2 + var.unsqueeze(-1))
    r = torch.exp(-0.5 * ((m.unsqueeze(-1) - bm) / s) ** 2) / (2 * torch.pi) ** 0.5 / s
    want = (r @ V64).transpose(1, 2).reshape(Bv, Q, D)
    e_tc, e_f = relerr(ctx, want), relerr(ctx_f, want)
    assert relerr(mu.view(Bv, H, Q), m) < 1e-5 and relerr(sd.view(Bv, H, Q), var.sqrt()) < 1e-3
    assert e_tc < 1e-3 and e_tc < 2 * e_f + 2e-5, (e_tc, e_f)      # (peaky random softmax: both ~3e-4 from fp64)
    assert relerr(mu, mu_f) < 1e-5


def test_fold_sample_columns(dev):
    """Variant G: operator columns summed per drawn sticky bin == the gathered product, G^T [R[b_s] ; k] = A_v [R ; k]."""
    ops = _ops()
    g = torch.Generator().manual_seed(12)
    Bv, N, S, L, e = 3, 64, 512, 8, 96
    GT = torch.randn(N, S + L + 4, generator=g)[:, :S + L + 4].to(dev)        # row pitch > S + L
    b = torch.randint(0, 127, (Bv, S), generator=g).sort(dim=1).values.int().to(dev)
    A = ops.fold_sample_columns(GT, b, S, L)
    assert A.shape == (Bv, N, 128 + L)
    R = torch.randn(Bv, 128, e, generator=g).double().to(dev)
    k = torch.randn(Bv, L, e, generator=g).double().to(dev)
    xm = torch.gather(R, 1, b.long().unsqueeze(-1).expand(-1, -1, e))
    want = GT[:, :S + L].double() @ torch.cat([xm, k], 1)
    got = A.double() @ torch.cat([R, k], 1)
    assert relerr(got, want) < 1e-6
    assert torch.equal(A[:, :, 128:], GT[:, S:S + L].unsqueeze(0).expand(Bv, -1, -1))
    assert float(A[:, :, 127].abs().max()) == 0.0                 # bin 127 is never drawn


# ---------------------------------------------------------------------------------------- R7
@pytest.mark.parametrize("ncat,Bv,zeros,sort", [(127, 1, False, False), (127, 37, True, False),
                                                (128, 5, False, True), (128, 4, True, True)])
def test_resample_is_bit_exact(dev, ncat, Bv, zeros, sort):
    """Given identical (p, u): bins, positions and basis indices bit-exact (north_star)."""
    ops, T = _ops(), _tables()
    g = torch.Generator().manual_seed(ncat + Bv)
    p = torch.rand(Bv, ncat, generator=g) ** 3
    if zeros:
        p[:, ::5] = 0
    u = torch.rand(Bv, 512, dtype=torch.float64, generator=g)
    # a few uniforms exactly on CDF edges (ties must resolve like torch: first category with cdf >= u)
    cum = torch.cumsum(p[0], 0)
    cdf0 = (cum / cum[-1]).double()
    u[0, :8] = cdf0[[3, 10, 20, 50, 70, 90, 100, ncat - 1]]
    tab = T.rect_tables(8, 256, .75)
    bins = torch.from_numpy(tab.bins).to(dev)
    b2b = torch.from_numpy(tab.bin2basis).to(dev)
    want_b = O.inverse_cdf_sample(p, u)
    out = ops.resample(p.to(dev), u.to(dev), bins, b2b, normalize=False, sort=sort)
    assert torch.equal(out["b_draw"].cpu().long(), want_b)
    used = torch.sort(want_b, -1)[0] if sort else want_b
    assert torch.equal(out["b_used"].cpu().long(), used)
    assert torch.equal(out["ts"].cpu(), torch.from_numpy(tab.bins)[used])          # exact bin left edges
    assert torch.equal(out["idx"].cpu().long(), torch.from_numpy(tab.bin2basis).long()[used])
    assert torch.equal(out["p"].cpu(), p)


def test_resample_normalised_partials(dev):
    """parts > 1 + the reference's two p/sum(p) passes; draws must be consistent with the p it reports."""
    ops, T = _ops(), _tables()
    g = torch.Generator().manual_seed(3)
    part = torch.rand(6, 12, 127, generator=g)
    u = torch.rand(6, 512, dtype=torch.float64, generator=g)
    tab = T.rect_tables(8, 64, .75)
    out = ops.resample(part.to(dev), u.to(dev), torch.from_numpy(tab.bins).to(dev),
                       torch.from_numpy(tab.bin2basis).to(dev), normalize=True, sort=False)
    p = part.sum(1)
    p = p / p.sum(-1, keepdim=True)
    p = p / p.sum(-1, keepdim=True)
    assert relerr(out["p"], p) < 1e-6
    assert torch.equal(out["b_draw"].cpu().long(), O.inverse_cdf_sample(out["p"].cpu(), u))


# ---------------------------------------------------------------------------------------- R6 / R10 / R11
def _rect_case(N, L, Q, seed, q_scale):
    key, val = make_proj(seed, 768)
    orc = O.RectLTM(N, .75, *proj_tensors(key, val), rebuild_tables=False)
    ks, qs, us = make_inputs(seed + 1, 1, 2, L * 32, 768, Q, q_scale)
    with torch.no_grad():
        outs = []
        for v in range(2):
            o = O.RectLTM(N, .75, *proj_tensors(key, val), rebuild_tables=False)
            ctx = o.forward(ks[0][v:v + 1], qs[0][v:v + 1], True)
            outs.append((o, ctx))
    return key, val, ks[0], qs[0], outs


def _tf32_rna(x):
    """Round-to-nearest (ties away) onto the tf32 grid, like cvt.rna.tf32.f32."""
    b = x.contiguous().view(torch.int32)
    return ((b + 0x1000) & ~0x1FFF).view(torch.float32)


@pytest.mark.parametrize("N,L,Q,q_scale", [(64, 8, 32, 1.0), (256, 16, 32, 8.0), (512, 16, 32, 4.0),
                                           (64, 8, 96, 2.0), (100, 30, 40, 2.0), (128, 16, 32, 2.0),
                                           (256, 8, 40, 1.0), (512, 32, 72, 1.0)])
def test_cont_attn_rect_and_fused_histogram(dev, N, L, Q, q_scale):
    ops, T = _ops(), _tables()
    key, val, k, q, outs = _rect_case(N, L, Q, 7, q_scale)
    tab = T.rect_tables(L, N, .75)
    td = tab.to(dev)
    Wkv = torch.cat([key.weight, val.weight]).detach()
    bkv = torch.cat([key.bias, val.bias]).detach()
    B = torch.cat([o.B_past for o, _ in outs])                                   # [2,N,e]
    KV = torch.nn.functional.linear(B, Wkv, bkv)                                 # fp32 CPU projection
    ctx, scores, hist = ops.cont_attn_rect(q.to(dev), KV.to(dev), td["W"], tab.W_out, td["jb"], td["tb"],
                                           want_scores=True, want_hist=True)
    want_ctx = torch.cat([c for _, c in outs])
    want_S = torch.cat([o.last["scores"] for o, _ in outs])
    assert relerr(scores, want_S) < 1e-5
    assert relerr(ctx, want_ctx) < 1e-4
    # fused sticky histogram == what the oracle would compute at the *next* call (gibbs:196-203)
    want_p = torch.cat([o.sticky_hist(o.tables(L)) for o, _ in outs])
    bins = td["bins"]
    u = torch.rand(2, 512, dtype=torch.float64).to(dev)
    got = ops.resample(hist, u, bins, td["bin2basis"], normalize=True)
    assert relerr(got["p"], want_p) < 2e-5
    # the standalone histogram op agrees with the fused one
    hp = ops.sticky_hist_rect(scores, td["jb"], td["tb"])
    got2 = ops.resample(hp, u, bins, td["bin2basis"], normalize=True)
    assert relerr(got2["p"], got["p"]) < 1e-5
    # transposed-key fast path (same inputs, K handed over as Kt[v][h][d][j])
    if ops.attn_fast_supported(N):
        Kt = KV[:, :, :768].reshape(2, N, 12, 64).permute(0, 2, 3, 1).contiguous()
        Vv = KV[:, :, 768:].contiguous()
        ctx3, scores3, hist3 = ops.cont_attn_rect_t(q.to(dev), Kt.to(dev), Vv.to(dev), td["W"], tab.W_out, td["jb"],
                                                     td["tb"], want_scores=True, want_hist=True)
        assert relerr(scores3, want_S) < 1e-5
        assert relerr(ctx3, want_ctx) < 1e-4
        got3 = ops.resample(hist3, u, bins, td["bin2basis"], normalize=True)
        assert relerr(got3["p"], want_p) < 2e-5
        ctx4, _, _ = ops.cont_attn_rect_t(q.to(dev), Kt.to(dev), Vv.to(dev), td["W"], tab.W_out, want_hist=False)
        assert torch.equal(ctx4, ctx3)
    # tensor-core path: both contractions as tf32 UMMAs over tf32-rounded K|V (tolerances are tf32's: operands carry
    # 2^-12 relative rounding; the scores enter an exponential, so ctx / p are held to 1e-3 like the e2e tests)
    if ops.attn_tc_supported(N) or ops.attn_tc_split_supported(N):     # (512: two basis halves + combine)
        KVr = _tf32_rna(KV).to(dev)
        ctx5, scores5, hist5 = ops.cont_attn_rect_tc(q.to(dev), KVr, td["X"], td["W"], tab.W_out, tab.c_none,
                                                     td["jb"], td["tb"], want_scores=True, want_hist=True)
        assert relerr(scores5, want_S) < 5e-4
        assert relerr(ctx5, want_ctx) < 1e-3
        got5 = ops.resample(hist5, u, bins, td["bin2basis"], normalize=True)
        assert relerr(got5["p"], want_p) < 1e-3
        ctx6, _, _ = ops.cont_attn_rect_tc(q.to(dev), KVr, td["X"], td["W"], tab.W_out, tab.c_none, want_hist=False)
        assert torch.equal(ctx6, ctx5)
        # fp16 K|V (kind::f16 UMMAs): the same 11-bit significand, same tolerances
        KVh = KV.half().to(dev)
        ctx7, scores7, hist7 = ops.cont_attn_rect_tc16(q.to(dev), KVh, td["X16"], td["W"], tab.W_out, tab.c_none,
                                                       td["jb"], td["tb"], want_scores=True, want_hist=True)
        assert relerr(scores7, want_S) < 5e-4
        assert relerr(ctx7, want_ctx) < 1e-3
        got7 = ops.resample(hist7, u, bins, td["bin2basis"], normalize=True)
        assert relerr(got7["p"], want_p) < 1e-3


# ---------------------------------------------------------------------------------------- R3/R5/R8
@pytest.mark.parametrize("N,L,tau,splits", [(64, 8, .75, 1), (256, 32, .75, 2), (100, 30, .5, 1), (64, 7, .75, 3)])
def test_consolidate_rect(dev, N, L, tau, splits):
    ops, T = _ops(), _tables()
    g = torch.Generator().manual_seed(N + L)
    Bv, e = 3, 768
    x = torch.randn(Bv, L, e, generator=g)
    B_past = torch.randn(Bv, N, e, generator=g)
    tab = T.rect_tables(L, N, tau)
    td = tab.to(dev)
    b = torch.randint(0, 127, (Bv, 512), generator=g)
    idx = torch.from_numpy(tab.bin2basis).long()[b]
    # split x into partial sums
    w = torch.rand(splits, generator=g)
    w = w / w.sum()
    xpart = torch.stack([x * w[s] for s in range(splits)], 2).contiguous()
    # first chunk: B = G0^T x
    want0 = torch.matmul(x.transpose(1, 2), torch.from_numpy(tab.dense_G0())).permute(0, 2, 1)
    got0 = ops.consolidate_rect(None, xpart.to(dev), None, None, td, 512)
    assert relerr(got0, want0) < 2e-6
    # update: B = G_inf^T [B_past[idx] ; x]
    xm = torch.stack([torch.where((idx[v] >= 0).unsqueeze(1), B_past[v][idx[v].clamp(min=0)],
                                  torch.zeros(1)) for v in range(Bv)])
    xcat = torch.cat([xm, x], 1)
    want1 = torch.matmul(xcat.transpose(1, 2), torch.from_numpy(tab.dense_Ginf())).permute(0, 2, 1)
    got1 = ops.consolidate_rect(B_past.to(dev), xpart.to(dev), idx.int().to(dev), None, td, 512)
    assert relerr(got1, want1) < 2e-6
    # per-video new_doc flags select the table set
    flags = torch.tensor([0, 1, 0], dtype=torch.uint8)
    got2 = ops.consolidate_rect(B_past.to(dev), xpart.to(dev), idx.int().to(dev), flags.to(dev), td, 512).cpu()
    assert torch.equal(got2[1], got0[1].cpu()) and torch.equal(got2[0], got1[0].cpu())


@pytest.mark.parametrize("N,L,tau,shared_idx", [(256, 64, .75, False), (64, 8, .75, False), (512, 32, .75, False),
                                                (100, 30, .5, False), (64, 8, .75, True)])
def test_consolidate_rect_carries_projected_memory(dev, N, L, tau, shared_idx):
    """Projected-memory state: K|V of the bins below `jf` from the previous K|V == projection of the new coefficients
    (the projection is affine, the contraction linear); rows >= jf are not touched."""
    ops, T = _ops(), _tables()
    g = torch.Generator().manual_seed(3 * N + L)
    Bv, e, D2 = 3, 768, 1536
    x = torch.randn(Bv, L, 1, e, generator=g)
    B_past = torch.randn(Bv, N, e, generator=g)
    W = torch.randn(D2, e, generator=g) / 28
    bias = torch.randn(D2, generator=g)
    KV_past = (B_past.double() @ W.double().t() + bias.double()).float()
    tab = T.rect_tables(L, N, tau)
    td = tab.to(dev)
    jf = tab.jf
    assert 0 < jf < N
    if shared_idx:
        idx = torch.from_numpy(tab.idx_uniform).int()
    else:
        b = torch.randint(0, 127, (Bv, 512), generator=g)
        idx = torch.from_numpy(tab.bin2basis)[b].int()
    B_new, KV_new = ops.consolidate_rect_kv(B_past.to(dev), x.to(dev), idx.to(dev), td, 512, KV_past.to(dev),
                                            bias.to(dev), jf)
    want_B = ops.consolidate_rect(B_past.to(dev), x.to(dev),
                                  (idx if idx.dim() == 2 else idx.expand(Bv, 512).contiguous()).to(dev), None, td, 512)
    assert torch.equal(B_new, want_B)
    want_KV = (B_new.double().cpu() @ W.double().t() + bias.double()).float()
    assert relerr(KV_new[:, :jf], want_KV[:, :jf]) < 2e-6
    assert float(KV_new[:, jf:].abs().max()) == 0.0
    # rounded store: every value on the tf32 grid, within half a tf32 ulp of the exact one
    _, KV_r = ops.consolidate_rect_kv(B_past.to(dev), x.to(dev), idx.to(dev), td, 512, KV_past.to(dev), bias.to(dev),
                                      jf, round_tf32=True)
    assert int((KV_r.view(torch.int32) & 0x1FFF).abs().max()) == 0
    assert relerr(KV_r[:, :jf], want_KV[:, :jf]) < 5e-4           # half a tf32 ulp = 2^-11 relative


def test_gemm_fp16_output_and_fp16_projected_memory(dev):
    """`c_fp16`: the GEMM epilogue stores IEEE fp16 (through the plain and the two-level row mapping); and the
    consolidation carries fp16 K|V rows (fp32 accumulation, one rounding at the store)."""
    ops, T = _ops(), _tables()
    g = torch.Generator().manual_seed(5)
    M, K, Nc = 300, 96, 160
    A = torch.randn(M, K, generator=g).to(dev)
    Bm = torch.randn(Nc, K, generator=g).to(dev)
    bias = torch.randn(Nc, generator=g).to(dev)
    Ch = torch.zeros(M, Nc, device=dev, dtype=torch.float16)
    ops.gemm_raw(A, K, 0, True, Bm, K, 0, True, Ch, Nc, 0, M, Nc, K, 1, bias=bias, precision="tf32", c_fp16=True)
    want = (A.double() @ Bm.double().t() + bias.double())
    assert relerr(Ch.float(), want) < 2e-3                      # single-pass TF32 product + one fp16 rounding
    C32 = torch.zeros(M, Nc, device=dev)
    ops.gemm_raw(A, K, 0, True, Bm, K, 0, True, C32, Nc, 0, M, Nc, K, 1, bias=bias, precision="tf32")
    assert torch.equal(Ch, C32.half())                          # the same accumulator, rounded once
    # two-level row mapping of A and C
    Cg = torch.zeros(5, 64, 160, device=dev, dtype=torch.float16)
    Ag = torch.randn(5, 64, K, generator=g).to(dev)
    ops.gemm_raw(Ag, K, 0, True, Bm, K, 0, True, Cg, Nc, 0, 5 * 32, Nc, K, 1, bias=bias, a_offset=32 * K, a_group=32,
                 a_group_stride=64 * K, c_offset=32 * Nc, c_group=32, c_group_stride=64 * Nc, c_fp16=True)
    assert float(Cg[:, :32].abs().max()) == 0.0
    assert relerr(Cg[:, 32:].float(), Ag[:, 32:].double() @ Bm.double().t() + bias.double()) < 2e-3
    # carried rows in fp16
    N, L, Bv, e, D2 = 256, 64, 2, 768, 1536
    tab = T.rect_tables(L, N, .75)
    td = tab.to(dev)
    x = torch.randn(Bv, L, 1, e, generator=g)
    B_past = torch.randn(Bv, N, e, generator=g)
    W = torch.randn(D2, e, generator=g) / 28
    bkv = torch.randn(D2, generator=g)
    KV_past = (B_past.double() @ W.double().t() + bkv.double()).half()
    idx = torch.from_numpy(tab.bin2basis)[torch.randint(0, 127, (Bv, 512), generator=g)].int()
    import ctypes as C
    from infinite_video_b200 import _capi
    B_new = torch.empty(Bv, N, e, device=dev)
    KV_new = torch.zeros(Bv, N, D2, device=dev, dtype=torch.float16)
    Bp, xp, ix, kvp, bk = B_past.to(dev), x.to(dev), idx.to(dev), KV_past.to(dev), bkv.to(dev)
    _capi.check(_capi.lib().ltm_consolidate_rect_kv(
        _capi.ptr(Bp), _capi.ptr(xp), _capi.ptr(ix), 512, None, _capi.ptr(td["seg_ptr0"]), _capi.ptr(td["seg_mem0"]),
        _capi.ptr(td["g0"]), _capi.ptr(td["seg_ptr1"]), _capi.ptr(td["seg_mem1"]), _capi.ptr(td["g1"]),
        _capi.ptr(B_new), None, _capi.ptr(kvp), _capi.ptr(KV_new), _capi.ptr(bk), D2, tab.jf, 2, Bv, N, e, L, 1, 512,
        _capi.stream_ptr(dev)), "consolidate_rect_kv")
    # reference: the same segmented mean over the fp16 rows in exact arithmetic
    Bn64, KVn = ops.consolidate_rect_kv(Bp, xp, ix, td, 512, kvp.float(), bk, tab.jf)
    assert torch.equal(B_new, Bn64)
    assert relerr(KV_new[:, :tab.jf].float(), KVn[:, :tab.jf]) < 6e-4
    assert float(KV_new[:, tab.jf:].abs().max()) == 0.0


@pytest.mark.parametrize("group,groups,N_rows", [(64, 6, 256), (16, 20, 64), (128, 3, 512), (256, 2, 1024), (32, 5, 40)])
@pytest.mark.parametrize("precision", ["tf32", "tf32x3"])
def test_gemm_grouped_rows(dev, group, groups, N_rows, precision):
    """A rows addressed in groups (rows [jf, N) of every video as one flat problem, one TMA box spanning several
    videos) and C written through the matching two-level mapping; checked against the SIMT kernel."""
    ops = _ops()
    g = torch.Generator().manual_seed(group + groups)
    K, Nc = 96, 160
    A = torch.randn(groups, N_rows, K, generator=g).to(dev)
    Bm = torch.randn(Nc, K, generator=g).to(dev)
    bias = torch.randn(Nc, generator=g).to(dev)
    j0 = N_rows - group
    outs = []
    for impl in ("tcgen05", "simt"):
        Cm = torch.zeros(groups, N_rows, Nc, device=dev)
        ops.gemm_raw(A, K, 0, True, Bm, K, 0, True, Cm, Nc, 0, groups * group, Nc, K, 1, bias=bias,
                     a_offset=j0 * K, a_group=group, a_group_stride=N_rows * K, c_offset=j0 * Nc,
                     c_group=group, c_group_stride=N_rows * Nc, precision=precision, impl=impl)
        outs.append(Cm)
    want = A[:, j0:].double() @ Bm.double().t() + bias.double()
    assert float(outs[0][:, :j0].abs().max()) == 0.0
    assert relerr(outs[1][:, j0:], want) < 1e-5
    assert relerr(outs[0][:, j0:], want) < (2e-3 if precision == "tf32" else 2e-5)


# ---------------------------------------------------------------------------------------- GEMM (tcgen05)
GEMM_CASES = [
    # M, N, K, batch, a_kmajor, b_kmajor, two_segment, bias
    (128, 128, 32, 1, True, True, False, False),       # one tile, one k-block
    (128, 128, 256, 1, True, True, False, True),
    (256, 1536, 768, 1, True, True, False, True),      # K/V projection shape (per 256 coefficient rows)
    (100, 72, 40, 1, True, True, False, False),        # ragged tails everywhere
    (384, 1536, 768, 1, True, True, False, True),      # odd number of row tiles
    (300, 520, 64, 2, True, True, False, True),        # ragged tails in M and N, batched, bias
    (1152, 256, 96, 1, False, True, False, False),     # A MN-major, B K-major, nine row tiles
    (128, 768, 256, 3, True, False, False, False),     # Psi_tab @ B_past[v]   (B MN-major, batched)
    (256, 768, 544, 2, True, False, True, False),      # G_inf^T [xm ; k]      (two K segments)
    (64, 768, 8, 2, True, False, False, False),        # G0^T k with Lk = 8
    (128, 256, 96, 2, False, True, False, False),      # A MN-major
    (96, 160, 64, 2, False, False, False, True),
]


@pytest.mark.parametrize("M,N,K,batch,akm,bkm,two,bias", GEMM_CASES)
@pytest.mark.parametrize("precision", ["tf32", "tf32x3"])
def test_gemm_tcgen05(dev, M, N, K, batch, akm, bkm, two, bias, precision):
    ops = _ops()
    g = torch.Generator().manual_seed(M * 7 + N + K)
    A = torch.randn(*((M, K) if akm else (K, M)), generator=g)                  # shared across the batch
    K1 = 32 * ((K // 2) // 32) if two else K
    Bfull = torch.randn(batch, *((N, K) if bkm else (K, N)), generator=g)
    bias_t = torch.randn(N, generator=g) if bias else None
    Am = A if akm else A.t()
    Bm = Bfull.transpose(1, 2) if bkm else Bfull                                  # [batch,K,N]
    want = torch.matmul(Am.double(), Bm.double())
    if bias:
        want = want + bias_t.double()
    if two:
        B1 = (Bfull[:, :, :K1] if bkm else Bfull[:, :K1]).contiguous()
        B2 = (Bfull[:, :, K1:] if bkm else Bfull[:, K1:]).contiguous()
    else:
        B1, B2 = Bfull, None
    got = ops.gemm(A.to(dev), B1.to(dev), B2=None if B2 is None else B2.to(dev), a_kmajor=akm, b_kmajor=bkm,
                   bias=None if bias_t is None else bias_t.to(dev), precision=precision, impl="tcgen05")
    tol = 3e-3 if precision == "tf32" else 2e-5
    assert relerr(got, want) < tol
    chk = ops.gemm(A.to(dev), B1.to(dev), B2=None if B2 is None else B2.to(dev), a_kmajor=akm, b_kmajor=bkm,
                   bias=None if bias_t is None else bias_t.to(dev), precision=precision, impl="simt")
    assert relerr(chk, want) < 1e-5


def test_project_kv(dev):
    ops = _ops()
    key, val = make_proj(2, 768)
    g = torch.Generator().manual_seed(5)
    B = torch.randn(512, 768, generator=g) * 0.02
    Wkv = torch.cat([key.weight, val.weight]).detach()
    bkv = torch.cat([key.bias, val.bias]).detach()
    want = torch.nn.functional.linear(B.double(), Wkv.double(), bkv.double())
    assert relerr(ops.project_kv(B.to(dev), Wkv.to(dev), bkv.to(dev), "tf32"), want) < 1e-3
    assert relerr(ops.project_kv(B.to(dev), Wkv.to(dev), bkv.to(dev), "tf32x3"), want) < 1e-5
    # keys transposed per head / values compact (fast attention path): same numbers, different layout
    for N in (64, 256):
        for impl in ("tcgen05", "simt"):
            Kt, V = ops.project_kv_t(B.to(dev), Wkv.to(dev), bkv.to(dev), N, "tf32x3", impl)
            wk = want[:, :768].reshape(512 // N, N, 12, 64).permute(0, 2, 3, 1)
            assert relerr(Kt, wk) < 1e-5 and relerr(V.reshape(512, 768), want[:, 768:]) < 1e-5


# ---------------------------------------------------------------------------------------- variant G kernels
@pytest.mark.parametrize("Bv,N,Q,H,L", [(3, 256, 1, 12, 64), (2, 128, 96, 16, 16), (1, 256, 33, 8, 32),
                                        (5, 128, 32, 1, 16)])
def test_tensor_core_attention_shapes(dev, Bv, N, Q, H, L):
    """The tensor-core attention against the fp32 FMA kernel on identical (tf32-rounded) K|V for shapes the end-to-end
    cases do not reach: a single query, several / partial query tiles, 1, 8 and 16 heads."""
    ops, T = _ops(), _tables()
    g = torch.Generator().manual_seed(Bv * 1000 + N + Q + H)
    D = H * 64
    tab = T.rect_tables(L, N, .75)
    td = tab.to(dev)
    KVr = _tf32_rna(torch.randn(Bv, N, 2 * D, generator=g)).to(dev)
    q = (torch.randn(Bv, Q, D, generator=g) * 2).to(dev)
    Kt = KVr[:, :, :D].reshape(Bv, N, H, 64).permute(0, 2, 3, 1).contiguous()
    V = KVr[:, :, D:].contiguous()
    c0, s0, h0 = ops.cont_attn_rect_t(q, Kt, V, td["W"], tab.W_out, td["jb"], td["tb"], want_scores=True)
    c1, s1, h1 = ops.cont_attn_rect_tc(q, KVr, td["X"], td["W"], tab.W_out, tab.c_none, td["jb"], td["tb"],
                                       want_scores=True, n_heads=H)
    assert relerr(s1, s0) < 5e-4 and relerr(c1, c0) < 1e-3 and relerr(h1, h0) < 1e-3
    assert bool(torch.isfinite(c1).all())


@pytest.mark.parametrize("M,N,K", [(512, 1536, 768), (300, 200, 136), (128, 256, 64)])
def test_gemm_fp16_operands(dev, M, N, K):
    """kind::f16 path of the tcgen05 GEMM: fp16 operands are exact inputs, products accumulate in fp32."""
    ops = _ops()
    g = torch.Generator().manual_seed(M + N + K)
    A = torch.randn(M, K, generator=g).half()
    B = (torch.randn(N, K, generator=g) * 0.05).half()
    bias = torch.randn(N, generator=g)
    want = A.double() @ B.double().t() + bias.double()
    got = ops.gemm_fp16(A.to(dev), B.to(dev), bias.to(dev))
    assert relerr(got, want.float()) < 2e-6


@pytest.mark.parametrize("M,N,K,batch", [(384, 768, 8192, 2), (128, 256, 64, 1), (300, 200, 136, 3), (96, 1024, 512, 1)])
def test_gemm_fp16_mn_major_b(dev, M, N, K, batch):
    """kind::f16 GEMM with the B operand MN-major (memory [K][N], 16-bit SWIZZLE_128B atoms of 8 k x 64 n): the value
    contraction of the short-term attention reads the fp16 chunk tokens this way (P[H*Q, LT] @ enc16[LT, e])."""
    ops = _ops()
    g = torch.Generator().manual_seed(M + N + K)
    A = (torch.rand(batch, M, K, generator=g) / K * 4).half().to(dev)             # probability-like rows
    B = torch.randn(batch, K, N, generator=g).half().to(dev)
    C = torch.zeros(batch, M, N, device=dev)
    ops.gemm_raw(A, K, M * K, True, B, N, K * N, False, C, N, M * N, M, N, K, batch, precision="tf32", ab_fp16=True)
    want = A.double() @ B.double()
    assert relerr(C, want) < 2e-5                        # exact fp16 products, fp32 accumulation over up to 8192 terms
    # K-major B through the same raw entry, and an fp16 result
    Bt = B.transpose(1, 2).contiguous()
    C2 = torch.zeros(batch, M, N, device=dev, dtype=torch.float16)
    ops.gemm_raw(A, K, M * K, True, Bt, K, N * K, True, C2, N, M * N, M, N, K, batch, precision="tf32", ab_fp16=True,
                 c_fp16=True)
    assert relerr(C2.float(), want) < 6e-4


def test_to_half_and_half_softmax(dev):
    ops = _ops()
    g = torch.Generator().manual_seed(9)
    x = torch.randn(3, 1000, 768, generator=g).to(dev)
    assert torch.equal(ops.to_half(x), x.half())
    S = (torch.randn(2, 40, 512, generator=g) * 3).to(dev)
    mask = torch.zeros(2, 512)
    mask[1, 400:] = -10000.0
    want = torch.softmax(S.cpu().double() * 0.125 + mask.double().unsqueeze(1), -1)
    P = ops.softmax_rows_half(S.clone(), 0.125, mask.to(dev), 40)
    assert P.dtype == torch.float16 and relerr(P.float(), want) < 6e-4
    assert float((P.float().sum(-1) - 1).abs().max()) < 2e-3
    # full rows of the caller's shape (register-resident kernel, n = 8192), a ragged width, and a row longer than the
    # registers hold (three-pass kernel)
    for n in (8192, 8188, 12288):
        S = (torch.randn(5, n, generator=g) * 4).to(dev)
        want = torch.softmax(S.cpu().double() * 0.125, -1)
        P = ops.softmax_rows_half(S.clone(), 0.125)
        assert relerr(P.float(), want) < 6e-4, n


def test_project_kv_rounded_to_tf32(dev):
    """`ltm_project_kv_r`: the same product as `ltm_project_kv`, stored on the tf32 grid (round to nearest)."""
    ops = _ops()
    torch.manual_seed(3)
    Bc = torch.randn(512, 768, device=dev)
    Wkv = torch.randn(1536, 768, device=dev) * 0.05
    bkv = torch.randn(1536, device=dev)
    plain = ops.project_kv(Bc, Wkv, bkv)
    rounded = ops.project_kv_r(Bc, Wkv, bkv)
    assert torch.equal(rounded, _tf32_rna(plain))
    assert int((rounded.view(torch.int32) & 0x1FFF).abs().max()) == 0


def test_rbf_eval_and_sticky_hist_gauss(dev):
    ops = _ops()
    psi = O.GaussBasis(256, [0.005, 0.01])
    t = torch.linspace(0, 1, 129)[:128]
    want = psi.at(t)
    got = ops.rbf_eval(t.to(dev), psi.mu[0].to(dev), psi.sigma[0].to(dev))
    assert relerr(got, want) < 1e-5
    g = torch.Generator().manual_seed(9)
    mu = torch.rand(3, 384, generator=g)
    sd = torch.rand(3, 384, generator=g) * 0.05 + 0.004
    key, val = make_proj(1, 768)
    orc = O.GaussLTM(256, .75, *proj_tensors(key, val))
    orc.attn_past = [mu, sd]
    bins, nudged = O.sticky_edges()
    want_p = orc.sticky_hist(dict(nudged=nudged))
    hist = ops.sticky_hist_gauss(mu.to(dev), sd.to(dev), nudged.to(dev))
    u = torch.rand(3, 512, dtype=torch.float64).to(dev)
    got = ops.resample(hist, u, bins.to(dev), None, normalize=True, sort=True)
    assert relerr(got["p"], want_p) < 1e-5


@pytest.mark.parametrize("N,L", [(64, 8), (256, 256)])
def test_ridge_solve_against_fp64(dev, N, L):
    """The device solver is checked against exact (fp64) arithmetic, not against the reference's fp32
    `.inverse()`, which is itself off by 1e-2 at this conditioning (SURVEY.md 0.5 / A7)."""
    ops, T = _ops(), _tables()
    t = T.gauss_tables(L, N, .75)
    mu, sg = torch.from_numpy(t.basis_mu), torch.from_numpy(t.basis_sigma)
    for pos, trim, rows in ((t.pos0, t.trim0, L), (t.pos1, t.trim1, 512 + L)):
        p = torch.from_numpy(pos).double()
        z = (p.unsqueeze(0) - mu.double().unsqueeze(1)) / sg.double().unsqueeze(1)
        F = torch.exp(-0.5 * z * z) / math.sqrt(2 * math.pi) / sg.double().unsqueeze(1)       # [N,P]
        A = F @ F.t() + 0.5 * torch.eye(N, dtype=torch.float64)
        G_true = torch.linalg.solve(A, F).t()[trim:trim + rows]                                # [rows,N]
        G, GT = ops.ridge_solve(torch.from_numpy(pos).to(dev), trim, rows, mu.to(dev), sg.to(dev), 0.5)
        assert relerr(G, G_true) < 1e-5
        assert torch.equal(GT.cpu(), G.cpu().t())
        # residual of the normal equations in fp64:  G (F F^T + ridge I) == F^T
        res = G.cpu().double() @ A - F.t()[trim:trim + rows]
        assert float(res.abs().max() / F.abs().max()) < 1e-5


def test_cont_attn_gauss(dev):
    ops = _ops()
    key, val = make_proj(4, 768)
    N, L, Bv = 256, 16, 2
    orc = O.GaussLTM(N, .75, *proj_tensors(key, val), rebuild_tables=False)
    ks, qs, _ = make_inputs(8, 1, Bv, L, 768, 32)
    with torch.no_grad():
        want = orc.forward(ks[0], qs[0], True)
    Wkv = torch.cat([key.weight, val.weight]).detach()
    bkv = torch.cat([key.bias, val.bias]).detach()
    KV = torch.nn.functional.linear(orc.B_past, Wkv, bkv)
    psi = orc.tables(L)["psi"]
    ctx, scores, mu, sd = ops.cont_attn_gauss(qs[0].to(dev), KV.to(dev), psi.mu[0].to(dev), psi.sigma[0].to(dev),
                                              want_scores=True)
    assert relerr(scores, orc.last["scores"]) < 1e-5
    assert relerr(mu, orc.attn_past[0]) < 1e-5
    assert relerr(sd, orc.attn_past[1]) < 1e-3       # var = E[t^2] - mu^2 cancels; see DESIGN.md
    assert relerr(ctx, want) < 1e-3
    Kt = KV[:, :, :768].reshape(Bv, N, 12, 64).permute(0, 2, 3, 1).contiguous()
    ctx2, scores2, mu2, sd2 = ops.cont_attn_gauss_t(qs[0].to(dev), Kt.to(dev), KV[:, :, 768:].contiguous().to(dev),
                                                    psi.mu[0].to(dev), psi.sigma[0].to(dev), want_scores=True)
    assert relerr(scores2, orc.last["scores"]) < 1e-5 and relerr(mu2, orc.attn_past[0]) < 1e-5
    assert relerr(sd2, orc.attn_past[1]) < 1e-3 and relerr(ctx2, want) < 1e-3
