"""Large-batch kernel paths against plain high-precision references.

Several kernels switch to another code path once the batch is large -- the batch the library is built for (128 videos
per GPU): 256-wide GEMM tiles, persistent attention CTAs that run several work items each, four coefficient rows per
consolidation CTA, a bounded pooling grid.  tests/test_gpu_kernels.py checks every entry point at 1-5 videos, where
none of these paths runs.  Here every test first asserts, with the host's own selection rule, that the large path is
the one taken, then compares the kernel with an fp64 evaluation on the device (every video, every row) and, where the
arithmetic of an item cannot depend on where it runs, with the same work done in another order or batch, bit for bit.
"""
import pytest
import torch

from oracle import ltm_oracle as O
from tests.helpers import make_inputs, make_proj, proj_tensors

pytestmark = pytest.mark.gpu

H, DH, D = 12, 64, 768
SENT = -77.0                      # sentinel of output positions a kernel must not touch (exact in fp16 and fp32)


@pytest.fixture(scope="module")
def dev(cuda_device):
    return cuda_device


@pytest.fixture(scope="module")
def sms(dev):
    return torch.cuda.get_device_properties(dev).multi_processor_count


def _ops():
    from infinite_video_b200 import ops
    return ops


def _tables():
    from infinite_video_b200 import tables
    return tables


def _gen(dev, seed):
    return torch.Generator(device=dev).manual_seed(seed)


def _relerr(a, b):
    """max |a - b| / max |b| in fp64 on the tensors' device (no copy of large tensors to the host)."""
    a, b = a.double(), b.double()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


def _relerr_rows(a, b):
    """Worst relative error over the leading dimension (videos / groups), each measured against its own maximum."""
    a, b = a.double().flatten(1), b.double().flatten(1)
    return float(((a - b).abs().amax(1) / b.abs().amax(1).clamp_min(1e-30)).max())


def _tf32_rna(x):
    """Round to nearest (ties away) onto the tf32 grid, like cvt.rna.tf32.f32."""
    b = x.contiguous().view(torch.int32)
    return ((b + 0x1000) & ~0x1FFF).view(torch.float32)


# ---------------------------------------------------------------------------------------- host selection rules
def _assert_gemm_256(M, Nc, batch):
    # gemm_tcgen05.cu:993-994  tiles256 = ceil(Nc/256) * ceil(M/128) * batch;  bn = (Nc > 128 && tiles256 >= 74) ? 256 : 128
    tiles256 = ((Nc + 255) // 256) * ((M + 127) // 128) * batch
    assert Nc > 128 and tiles256 >= 74, (M, Nc, batch, tiles256)


def _attn_slots(sms, nb_item):
    # attn_tc.cu launch()  PER_SM = (2 * Lay<NB, KV>::BYTES <= 227 KB) ? 2 : 1 -- two CTAs per SM for 64 / 128
    # bases per item (60 / 106 KB of shared memory), one for 256 (209 KB);  grid = min(items, num_sms * PER_SM)
    return sms * (2 if nb_item < 256 else 1)


def _assert_multi_item(items, slots):
    # attn_tc.cu launch() / attn_g16.cu launch()  grid = min(total, slots): CTA b runs items b, b + grid, ...
    assert items >= 2 * slots and items % slots != 0, (items, slots)


def _assert_four_rows(N, Bv):
    # consolidate.cu:267  rows_per_cta = (N >= 128 && N * Bv >= 16384) ? 4 : 1
    assert N >= 128 and N * Bv >= 16384, (N, Bv)


def _assert_one_row(N, Bv):
    assert not (N >= 128 and N * Bv >= 16384), (N, Bv)


# ---------------------------------------------------------------------------------------- A. GEMM, 256-wide tiles
@pytest.mark.parametrize("groups", [128, 127])
def test_update_projection_grouped_rows(dev, groups):
    """K/V projection of an update chunk: rows [192, 256) of every video (a_group 64, one 128-row TMA box spans two
    videos; 127 videos leave the last box half filled), fp16 operands, fp16 output through the two-level C mapping."""
    ops = _ops()
    g = _gen(dev, 100 + groups)
    N, j0, grp, K, Nc = 256, 192, 64, 768, 1536
    M = groups * grp
    _assert_gemm_256(M, Nc, 1)
    A = torch.randn(groups, N, K, device=dev, generator=g).half()
    W = (torch.randn(Nc, K, device=dev, generator=g) / 28).half()
    bias = torch.randn(Nc, device=dev, generator=g)
    kw = dict(bias=bias, a_offset=j0 * K, a_group=grp, a_group_stride=N * K, c_offset=j0 * Nc, c_group=grp,
              c_group_stride=N * Nc, ab_fp16=True, precision="tf32")
    outs = []
    for max_ctas in (0, 64, 7):
        Ch = torch.full((groups, N, Nc), SENT, device=dev, dtype=torch.float16)
        ops.gemm_raw(A, K, 0, True, W, K, 0, True, Ch, Nc, 0, M, Nc, K, 1, c_fp16=True, max_ctas=max_ctas, **kw)
        outs.append(Ch)
    for o in outs[1:]:
        assert torch.equal(o, outs[0])                       # a bounded persistent grid walks the same tiles
    C32 = torch.full((groups, N, Nc), SENT, device=dev)
    ops.gemm_raw(A, K, 0, True, W, K, 0, True, C32, Nc, 0, M, Nc, K, 1, **kw)
    assert bool((outs[0][:, :j0] == SENT).all()) and bool((C32[:, :j0] == SENT).all())
    assert torch.equal(outs[0][:, j0:], C32[:, j0:].half())     # the same accumulator, rounded once
    want = A[:, j0:].double() @ W.double().t() + bias.double()
    assert _relerr_rows(C32[:, j0:], want) < 2e-6


def test_first_chunk_projection_full_height(dev):
    """First chunk of 128 videos x 256 coefficient rows in one plain GEMM, fp16 operands and output."""
    ops = _ops()
    g = _gen(dev, 101)
    M, K, Nc = 128 * 256, 768, 1536
    _assert_gemm_256(M, Nc, 1)
    A = torch.randn(M, K, device=dev, generator=g).half()
    W = (torch.randn(Nc, K, device=dev, generator=g) / 28).half()
    bias = torch.randn(Nc, device=dev, generator=g)
    Ch = torch.empty(M, Nc, device=dev, dtype=torch.float16)
    C32 = torch.empty(M, Nc, device=dev)
    ops.gemm_raw(A, K, 0, True, W, K, 0, True, Ch, Nc, 0, M, Nc, K, 1, bias=bias, ab_fp16=True, c_fp16=True)
    ops.gemm_raw(A, K, 0, True, W, K, 0, True, C32, Nc, 0, M, Nc, K, 1, bias=bias, ab_fp16=True)
    assert torch.equal(Ch, C32.half())
    want = A.double() @ W.double().t() + bias.double()
    assert _relerr_rows(C32.view(128, -1), want.view(128, -1)) < 2e-6


def test_fp32_operands_on_256_wide_tiles(dev):
    """fp32 operands: single-pass tf32, tf32 with the result rounded onto the tf32 grid, and split-TF32."""
    ops = _ops()
    g = _gen(dev, 102)
    M, K, Nc = 8192, 768, 1536
    _assert_gemm_256(M, Nc, 1)
    A = torch.randn(M, K, device=dev, generator=g)
    W = torch.randn(Nc, K, device=dev, generator=g) / 28
    bias = torch.randn(Nc, device=dev, generator=g)
    want = A.double() @ W.double().t() + bias.double()
    out = {}
    for name, prec, rnd in (("tf32", "tf32", False), ("rounded", "tf32", True), ("x3", "tf32x3", False)):
        out[name] = torch.empty(M, Nc, device=dev)
        ops.gemm_raw(A, K, 0, True, W, K, 0, True, out[name], Nc, 0, M, Nc, K, 1, bias=bias, precision=prec,
                     round_tf32=rnd)
    assert _relerr(out["tf32"], want) < 3e-3
    assert torch.equal(out["rounded"], _tf32_rna(out["tf32"]))
    assert int((out["rounded"].view(torch.int32) & 0x1FFF).abs().max()) == 0
    assert _relerr(out["x3"], want) < 2e-5
    few = torch.empty(M, Nc, device=dev)
    ops.gemm_raw(A, K, 0, True, W, K, 0, True, few, Nc, 0, M, Nc, K, 1, bias=bias, precision="tf32x3", max_ctas=7)
    assert torch.equal(few, out["x3"])


def test_ragged_problem(dev):
    """M = 10000 (partial last row tile), Nc = 1004 (the fp16 epilogue's scalar column tail; the row pitch 1008 keeps
    the other columns on 16-byte stores), K = 200 (a partial k-block in both operand formats)."""
    ops = _ops()
    g = _gen(dev, 103)
    M, Nc, K, ldc = 10000, 1004, 200, 1008
    _assert_gemm_256(M, Nc, 1)
    A = torch.randn(M, K, device=dev, generator=g)
    W = torch.randn(Nc, K, device=dev, generator=g) / 14
    bias = torch.randn(Nc, device=dev, generator=g)
    A16, W16 = A.half(), W.half()
    Ch = torch.full((M, ldc), SENT, device=dev, dtype=torch.float16)
    C32 = torch.full((M, ldc), SENT, device=dev)
    ops.gemm_raw(A16, K, 0, True, W16, K, 0, True, Ch, ldc, 0, M, Nc, K, 1, bias=bias, ab_fp16=True, c_fp16=True)
    ops.gemm_raw(A16, K, 0, True, W16, K, 0, True, C32, ldc, 0, M, Nc, K, 1, bias=bias, ab_fp16=True)
    assert bool((Ch[:, Nc:] == SENT).all()) and bool((C32[:, Nc:] == SENT).all())
    assert torch.equal(Ch[:, :Nc], C32[:, :Nc].half())
    assert _relerr(C32[:, :Nc], A16.double() @ W16.double().t() + bias.double()) < 2e-6
    X3 = torch.full((M, ldc), SENT, device=dev)
    ops.gemm_raw(A, K, 0, True, W, K, 0, True, X3, ldc, 0, M, Nc, K, 1, bias=bias, precision="tf32x3")
    assert bool((X3[:, Nc:] == SENT).all())
    assert _relerr(X3[:, :Nc], A.double() @ W.double().t() + bias.double()) < 2e-5


@pytest.mark.parametrize("layout", ["batch", "group"])
def test_fp16_output_with_unaligned_batch_or_group_stride(dev, layout):
    """fp16 output whose batch stride (or group stride) is 4 mod 8 halves: every other batch / group starts 8 bytes
    off a 16-byte boundary, so the epilogue must store its halves one by one there (two-term output included)."""
    ops = _ops()
    g = _gen(dev, 104)
    Nc, K, ldc = 768, 256, 768
    if layout == "batch":
        batch, M = 3, 1200
        stride = M * ldc + 4
        shape, span = (batch, M, Nc), batch * stride
        A = torch.randn(batch, M, K, device=dev, generator=g).half()
        lay, lay32 = dict(strideC=stride, batch=batch), dict(strideC=M * Nc, batch=batch)
        strideA, Mrun = M * K, M
    else:
        groups, grp = 64, 64
        batch, M = 1, groups * grp
        stride = grp * ldc + 4
        shape, span = (groups, grp, Nc), groups * stride
        A = torch.randn(M, K, device=dev, generator=g).half()
        lay = dict(strideC=0, batch=1, c_group=grp, c_group_stride=stride)
        lay32 = dict(strideC=0, batch=1)
        strideA, Mrun = 0, M
    assert stride % 8 == 4 and stride % 4 == 0
    _assert_gemm_256(Mrun, Nc, batch)
    W = (torch.randn(Nc, K, device=dev, generator=g) / 16).half()
    bias = torch.randn(Nc, device=dev, generator=g)
    hi = torch.full((span + 8,), SENT, device=dev, dtype=torch.float16)
    lo = torch.full((span + 8,), SENT, device=dev, dtype=torch.float16)

    def run(Cbuf, ldc_, c_fp16, C_lo, lay_):
        extra = {k: v for k, v in lay_.items() if k not in ("strideC", "batch")}
        ops.gemm_raw(A, K, strideA, True, W, K, 0, True, Cbuf, ldc_, lay_["strideC"], Mrun, Nc, K, lay_["batch"],
                     bias=bias, ab_fp16=True, c_fp16=c_fp16, C_lo=C_lo, precision="tf32", **extra)

    run(hi, ldc, True, lo, lay)
    full = torch.empty(shape, device=dev)
    run(full, Nc, False, None, lay32)
    view_hi = hi.as_strided(shape, (stride, ldc, 1))
    view_lo = lo.as_strided(shape, (stride, ldc, 1))
    assert torch.equal(view_hi, full.half())
    assert torch.equal(view_lo, (full - view_hi.float()).half())
    touched = torch.zeros(span + 8, device=dev, dtype=torch.bool)
    touched.as_strided(shape, (stride, ldc, 1)).fill_(True)
    assert bool((hi[~touched] == SENT).all()) and bool((lo[~touched] == SENT).all())
    want = A.double().view(shape[0], -1, K) @ W.double().t() + bias.double()
    assert _relerr_rows(full, want) < 2e-6
    assert _relerr_rows(view_hi.float() + view_lo.float(), want) < 2e-6


def test_variant_g_production_gemms(dev):
    """The GEMMs of variant G at 128 videos x 256 bases: the K/V projection as one fp16 GEMM over hi/lo-split
    operands (keys stored transposed per head, and the two-term fp16 output), and the two state GEMMs
    Psi_tab B_past[v] (batched, MN-major B, split-TF32) and A_v [R ; k] (two K segments)."""
    ops, T = _ops(), _tables()
    g = _gen(dev, 105)
    Bv, N, e, L = 128, 256, 768, 64
    M = Bv * N
    _assert_gemm_256(M, 2 * D, 1)
    Bc = torch.randn(M, e, device=dev, generator=g) * 0.5
    Wkv = torch.randn(2 * D, e, device=dev, generator=g) / 28
    bkv = torch.randn(2 * D, device=dev, generator=g)
    want = Bc.double() @ Wkv.double().t() + bkv.double()
    Kt, V = ops.project_kv_t(Bc, Wkv, bkv, N, "fp16x2")
    assert _relerr_rows(Kt, want[:, :D].reshape(Bv, N, H, DH).permute(0, 2, 3, 1)) < 1e-5
    assert _relerr_rows(V, want[:, D:].reshape(Bv, N, D)) < 1e-5
    hi, lo = ops.project_kv_split(Bc, bkv, N, ops.split_half3(Wkv, 1))
    assert _relerr_rows(hi.float() + lo.float(), want.view(Bv, N, 2 * D)) < 1e-5
    # Psi_tab [128 sticky positions, N] @ B_past[v] [N, e]
    t = T.gauss_tables(L, N, .75)
    psi = ops.rbf_eval(torch.from_numpy(t.bins[:128]).to(dev), torch.from_numpy(t.basis_mu).to(dev),
                       torch.from_numpy(t.basis_sigma).to(dev))
    B_past = torch.randn(Bv, N, e, device=dev, generator=g)
    _assert_gemm_256(128, e, Bv)
    R = ops.gemm(psi, B_past, b_kmajor=False, precision="tf32x3")
    assert _relerr_rows(R, psi.double() @ B_past.double()) < 2e-5
    # A_v [N, 128 + L] @ [R ; k]: the folded operator against the re-sampled rows and the chunk's frames
    Av = torch.randn(Bv, N, 128 + L, device=dev, generator=g)
    k = torch.randn(Bv, L, e, device=dev, generator=g)
    _assert_gemm_256(N, e, Bv)
    B_new = ops.gemm(Av, R, B2=k, b_kmajor=False, precision="tf32x3")
    assert _relerr_rows(B_new, Av.double() @ torch.cat([R, k], 1).double()) < 2e-5


# ---------------------------------------------------------------------------------------- B. attention, many items per CTA
def _rect_reference(q, KV, tab, tb=None):
    """fp64 closed form of the rectangular-basis attention: scores S = q_h K_h^T / sqrt(d), weights
    r_j = W_j e^{S_j} / (sum_i W_i e^{S_i} + W_out), ctx = r V, and the sticky histogram of the next call (the density
    e^{S} / trapz at the 129 nudged edges, trapezoid mass of the edge intervals 1..127, summed over heads and queries)."""
    Bv, Q, _ = q.shape
    N = KV.shape[1]
    dv = q.device
    qh = q.double().view(Bv, Q, H, DH).transpose(1, 2) / DH ** 0.5
    K = KV[:, :, :D].double().view(Bv, N, H, DH).transpose(1, 2)
    V = KV[:, :, D:].double().view(Bv, N, H, DH).transpose(1, 2)
    S = qh @ K.transpose(-1, -2)                                             # [Bv,H,Q,N]
    m = S.amax(-1, keepdim=True).clamp_min(0)                                # shift; cancels exactly
    W = torch.from_numpy(tab.W).double().to(dv)
    ew = W * torch.exp(S - m)
    r = ew / (ew.sum(-1, keepdim=True) + tab.W_out * torch.exp(-m))
    ctx = (r @ V).transpose(1, 2).reshape(Bv, Q, D)
    jb = torch.from_numpy(tab.jb).long().to(dv)
    tb = torch.from_numpy(tab.tb).double().to(dv) if tb is None else tb.double().to(dv)
    z = torch.where(jb >= 0, S[..., jb.clamp_min(0)], torch.zeros((), dtype=torch.float64, device=dv))
    ez = torch.exp(z - m)                                                    # [Bv,H,Q,129]
    seg = 0.5 * (ez[..., 1:] + ez[..., :-1]) * (tb[1:] - tb[:-1])           # [Bv,H,Q,128]
    dens = seg / seg.sum(-1, keepdim=True)                                   # / trapz over all edges
    p = dens[..., 1:].sum((1, 2))                                            # intervals 1..127 (gibbs:196-203)
    return S, ctx, p / p.sum(-1, keepdim=True)


def test_rect_reference_matches_the_oracle(monkeypatch):
    """The fp64 closed form above against the oracle module (faithful 1000-point quadrature, density by trapz) on
    two videos: the scores, the context and the sticky histogram.  The oracle runs in fp64 here (float64 default
    dtype; its indicator matrices, exact in any type, take the positions' dtype), so that what is compared is the
    formula, not the oracle's own fp32 rounding (3e-6 on the context)."""
    N, L, Q = 256, 16, 40
    key, val = make_proj(21, 768)
    ks, qs, _ = make_inputs(22, 1, 2, L * 32, 768, Q, 2.0)
    tab = _tables().rect_tables(L, N, .75)                    # (built, and cached, with fp32 positions as always)
    w = [t.double() for t in proj_tensors(key, val)]
    at = O.RectBasis.at
    monkeypatch.setattr(O.RectBasis, "at", lambda self, t: at(self, t).to(t.dtype))
    dtype = torch.get_default_dtype()
    torch.set_default_dtype(torch.float64)
    try:
        with torch.no_grad():
            for v in range(2):
                o = O.RectLTM(N, .75, *w, rebuild_tables=False)
                ctx = o.forward(ks[0][v:v + 1].double(), qs[0][v:v + 1].double(), True)
                KV = torch.nn.functional.linear(o.B_past, torch.cat([w[0], w[2]]), torch.cat([w[1], w[3]]))
                p = o.sticky_hist(o.tables(L))
                # (on the oracle's fp64 edges: the library's table holds them in fp32, 1.000001 -> 1.00000095)
                S, ctx64, p64 = _rect_reference(qs[0][v:v + 1], KV, tab, tb=o.tables(L)["nudged"])
                assert _relerr(o.last["scores"], S) < 1e-6
                assert _relerr(ctx, ctx64) < 1e-6
                assert _relerr(p, p64) < 1e-6
    finally:
        torch.set_default_dtype(dtype)


def _rect_tc(kind, q, KVk, tab, td):
    ops = _ops()
    if kind == "tc":
        return ops.cont_attn_rect_tc(q, KVk, td["X"], td["W"], tab.W_out, tab.c_none, td["jb"], td["tb"],
                                     want_scores=True, want_hist=True)
    return ops.cont_attn_rect_tc16(q, KVk, td["X16"], td["W"], tab.W_out, tab.c_none, td["jb"], td["tb"],
                                   want_scores=True, want_hist=True)


RECT_CASES = [(kind, N, 38, 40) for kind in ("tc16", "tc") for N in (64, 128, 256, 512)] + \
             [("tc16", 256, 128, 32), ("tc", 256, 128, 32)]          # (the headline batch: 128 videos, 32 queries)


@pytest.mark.parametrize("kind,N,Bv,Q", RECT_CASES)
def test_rect_attention_many_items_per_cta(dev, sms, kind, N, Bv, Q):
    """Tensor-core rectangular-basis attention with every CTA running several work items: each video against the fp64
    closed form, and the same items run in reverse order and alone give the same bits."""
    ops, T = _ops(), _tables()
    q_tiles = (Q + 31) // 32
    halves = 2 if N == 512 else 1                # num_basis 512: two basis halves + attn_tc_combine_kernel
    items = q_tiles * H * Bv * halves
    _assert_multi_item(items, _attn_slots(sms, N // halves))
    assert ops.attn_tc_supported(N) or ops.attn_tc_split_supported(N)
    tab = T.rect_tables(16, N, .75)
    td = tab.to(dev)
    g = _gen(dev, 200 + N + Bv)
    q = torch.randn(Bv, Q, D, device=dev, generator=g) * 2
    KV = torch.randn(Bv, N, 2 * D, device=dev, generator=g) * 0.5
    KVk = _tf32_rna(KV) if kind == "tc" else KV.half()                    # the kernel's operand format
    ctx, scores, hist = _rect_tc(kind, q, KVk, tab, td)
    S, ctx64, p64 = _rect_reference(q, KVk, tab)
    u = torch.rand(Bv, 512, dtype=torch.float64, device=dev, generator=g)
    p = ops.resample(hist, u, td["bins"], td["bin2basis"], normalize=True)["p"]
    assert _relerr_rows(scores, S) < 5e-4
    assert _relerr_rows(ctx, ctx64) < 1e-3
    assert _relerr_rows(p, p64) < 1e-3
    # item-position invariance: an item's arithmetic does not depend on which CTA runs it, nor in which iteration
    rc, rs, rh = _rect_tc(kind, q.flip(0).contiguous(), KVk.flip(0).contiguous(), tab, td)
    assert torch.equal(rc.flip(0), ctx) and torch.equal(rs.flip(0), scores) and torch.equal(rh.flip(0), hist)
    for v in (0, Bv // 2, Bv - 1):
        sc, ss, sh = _rect_tc(kind, q[v:v + 1].contiguous(), KVk[v:v + 1].contiguous(), tab, td)
        assert torch.equal(sc, ctx[v:v + 1]) and torch.equal(ss, scores[v:v + 1]) and torch.equal(sh, hist[v:v + 1])


def _gauss_reference(q, KV, bmu, bsig):
    """fp64 closed form of the Gaussian-basis attention (test_cont_attn_gauss_on_tensor_cores)."""
    Bv, Q, _ = q.shape
    N = KV.shape[1]
    K64 = KV[:, :, :D].double().view(Bv, N, H, DH).transpose(1, 2)
    V64 = KV[:, :, D:].double().view(Bv, N, H, DH).transpose(1, 2)
    qh = q.double().view(Bv, Q, H, DH).transpose(1, 2) / 8.0
    a = torch.softmax(20 * (qh @ K64.transpose(-1, -2)), -1)
    bm, bs = bmu.double(), bsig.double()
    m = a @ bm
    var = a @ (bm ** 2 + bs ** 2) - m ** 2
    s = torch.sqrt(bs ** 2 + var.unsqueeze(-1))
    r = torch.exp(-0.5 * ((m.unsqueeze(-1) - bm) / s) ** 2) / (2 * torch.pi) ** 0.5 / s
    return (r @ V64).transpose(1, 2).reshape(Bv, Q, D), m, var.sqrt()


@pytest.mark.parametrize("N,Bv,Q", [(256, 38, 40), (256, 128, 32)])
def test_gauss_attention_many_items_per_cta(dev, sms, N, Bv, Q):
    ops, T = _ops(), _tables()
    items = ((Q + 31) // 32) * H * Bv
    _assert_multi_item(items, sms)                            # attn_g16.cu:467: one CTA per SM
    t = T.gauss_tables(8, N, .75)
    bmu, bsig = torch.from_numpy(t.basis_mu).to(dev), torch.from_numpy(t.basis_sigma).to(dev)
    g = _gen(dev, 300 + N + Bv)
    q = torch.randn(Bv, Q, D, device=dev, generator=g)
    KV = torch.randn(Bv, N, 2 * D, device=dev, generator=g) * 0.5
    KV[:, :, D:] *= 3.0
    hi = KV.half()
    lo = (KV - hi.float()).half()
    ctx, mu, sd = ops.cont_attn_gauss_tc16(q, hi, lo, bmu, bsig)
    ctx64, m64, sd64 = _gauss_reference(q, KV, bmu, bsig)
    assert _relerr_rows(mu.view(Bv, H, Q), m64) < 1e-5
    assert _relerr_rows(sd.view(Bv, H, Q), sd64) < 1e-3
    assert _relerr_rows(ctx, ctx64) < 1e-3
    rc, rm, rs = ops.cont_attn_gauss_tc16(q.flip(0).contiguous(), hi.flip(0).contiguous(), lo.flip(0).contiguous(),
                                          bmu, bsig)
    assert torch.equal(rc.flip(0), ctx) and torch.equal(rm.flip(0), mu) and torch.equal(rs.flip(0), sd)
    for v in (0, Bv // 2, Bv - 1):
        sc, sm_, ss = ops.cont_attn_gauss_tc16(q[v:v + 1].contiguous(), hi[v:v + 1].contiguous(),
                                               lo[v:v + 1].contiguous(), bmu, bsig)
        assert torch.equal(sc, ctx[v:v + 1]) and torch.equal(sm_, mu[v:v + 1]) and torch.equal(ss, sd[v:v + 1])


# ---------------------------------------------------------------------------------------- C. consolidation, 4 rows per CTA
def _capi():
    from infinite_video_b200 import _capi
    return _capi


def _consolidate_kv16(B_past, xpart, idx, idx_stride, flags, td, tab, KV_past, bkv, S):
    """ltm_consolidate_rect_kv with fp16 K|V (round_tf32 = 2) and the fp16 copy of B: -> (B_new, B_half, KV_new), the
    two fp16 outputs pre-filled with the sentinel."""
    ca = _capi()
    Bv, L, splits, e = xpart.shape
    N = tab.N
    B_new = torch.empty(Bv, N, e, device=xpart.device)
    B_half = torch.full((Bv, N, e), SENT, device=xpart.device, dtype=torch.float16)
    KV_new = torch.full(KV_past.shape, SENT, device=xpart.device, dtype=torch.float16)
    ca.check(ca.lib().ltm_consolidate_rect_kv(
        ca.ptr(B_past), ca.ptr(xpart), ca.ptr(idx), idx_stride, ca.ptr(flags), ca.ptr(td["seg_ptr0"]),
        ca.ptr(td["seg_mem0"]), ca.ptr(td["g0"]), ca.ptr(td["seg_ptr1"]), ca.ptr(td["seg_mem1"]), ca.ptr(td["g1"]),
        ca.ptr(B_new), ca.ptr(B_half), ca.ptr(KV_past), ca.ptr(KV_new), ca.ptr(bkv), KV_past.shape[-1], tab.jf, 2, Bv, N,
        e, L, splits, S, ca.stream_ptr(xpart.device)), "consolidate_rect_kv")
    return B_new, B_half, KV_new


@pytest.mark.parametrize("N,Bv", [(256, 64), (512, 32), (128, 128), (134, 123)])     # (134: the last CTA has 2 rows)
def test_consolidation_four_rows_per_cta(dev, N, Bv):
    """Coefficients (first chunk, update, mixed new_doc flags, per-video and shared sample rows) against the dense fp64
    G^T [xm ; x]; the fp16 K|V rows below jf against the fp64 segmented mean; the fp16 copy of B; and the same videos
    consolidated as a batch of three (the one-row kernel, same summation order) give the same bits."""
    ops, T = _ops(), _tables()
    _assert_four_rows(N, Bv)
    S, L, e, splits, D2 = 512, 64, 768, 2, 1536
    tab = T.rect_tables(L, N, .75)
    td = tab.to(dev)
    assert 0 < tab.jf < N
    g = _gen(dev, 400 + N + Bv)
    xpart = torch.randn(Bv, L, splits, e, device=dev, generator=g)
    B_past = torch.randn(Bv, N, e, device=dev, generator=g)
    b = torch.randint(0, 127, (Bv, S), device=dev, generator=g)
    idx = td["bin2basis"][b].int().contiguous()
    flags = torch.zeros(Bv, device=dev, dtype=torch.uint8)
    flags[1::5] = 1
    bkv = torch.randn(D2, device=dev, generator=g)
    KV_past = (torch.randn(Bv, N, D2, device=dev, generator=g) * 0.5).half()
    G0 = torch.from_numpy(tab.dense_G0()).double().to(dev)                  # [L, N]
    Gi = torch.from_numpy(tab.dense_Ginf()).double().to(dev)                # [S + L, N]
    x = xpart.double().sum(2)                                               # [Bv, L, e]
    want0 = G0.t() @ x

    def want_update(ix):                                                    # ix: [Bv, S] (-1: no basis)
        valid = (ix >= 0).unsqueeze(-1)
        xm = torch.where(valid, torch.gather(B_past.double(), 1, ix.clamp_min(0).long().unsqueeze(-1).expand(-1, -1, e)),
                         torch.zeros((), dtype=torch.float64, device=dev))
        return Gi.t() @ torch.cat([xm, x], 1)

    def want_kv(ix):                                                        # rows j < jf: g sum KV_past[ix] + (1 - g cnt) b
        jf = tab.jf
        valid = (ix >= 0).double()
        rows = torch.gather(KV_past.double(), 1, ix.clamp_min(0).long().unsqueeze(-1).expand(-1, -1, D2))
        Gs = Gi[:S, :jf]                                                     # [S, jf]
        mass = (valid.unsqueeze(-1) * Gs).sum(1)                              # [Bv, jf] = g_j cnt_j
        return Gs.t() @ (rows * valid.unsqueeze(-1)) + (1 - mass).unsqueeze(-1) * bkv.double()

    got0 = ops.consolidate_rect(None, xpart, None, None, td, S)
    assert _relerr_rows(got0, want0) < 2e-6
    new = flags.bool().view(Bv, 1, 1)
    sel = torch.tensor([1, Bv // 2, Bv - 1], device=dev)                   # (video 1 starts a new document)
    _assert_one_row(N, 3)
    for mode in ("per_video", "shared"):
        if mode == "per_video":
            ix, ix_arg, stride = idx, idx, S
        else:                                     # the uniform re-sampling row, one for all videos (idx_stride 0)
            ix_arg = td["idx_uniform"]
            ix, stride = ix_arg.unsqueeze(0).expand(Bv, S).contiguous(), 0
        want1 = torch.where(new, want0, want_update(ix))
        got1 = ops.consolidate_rect(B_past, xpart, ix, flags, td, S)
        assert _relerr_rows(got1, want1) < 2e-6, mode
        Bn, Bh, KVn = _consolidate_kv16(B_past, xpart, ix_arg, stride, flags, td, tab, KV_past, bkv, S)
        assert torch.equal(Bn, got1), mode
        # fp16 K|V: rows below jf of continuing videos carried, everything else left to the projection
        cont = ~flags.bool()
        assert _relerr_rows(KVn[cont, :tab.jf].float(), want_kv(ix)[cont]) < 6e-4, mode
        assert bool((KVn[cont, tab.jf:] == SENT).all()) and bool((KVn[~cont] == SENT).all()), mode
        # fp16 copy of B on the rows the projection reads: new documents all rows, continuing videos rows >= jf
        read = new.expand(Bv, N, 1) | (torch.arange(N, device=dev) >= tab.jf).view(1, N, 1)
        assert torch.equal(torch.where(read, Bh, Bn.half()), Bn.half()), mode
        assert bool(torch.where(read, torch.full_like(Bh, SENT), Bh).eq(SENT).all()), mode
        # three videos alone: the one-row kernel, the same sums in the same order
        ix3 = ix_arg if stride == 0 else ix[sel].contiguous()
        sub = ops.consolidate_rect(B_past[sel].contiguous(), xpart[sel].contiguous(), ix[sel].contiguous(),
                                   flags[sel].contiguous(), td, S)
        assert torch.equal(sub, got1[sel]), mode
        B3, Bh3, KV3 = _consolidate_kv16(B_past[sel].contiguous(), xpart[sel].contiguous(), ix3, stride,
                                         flags[sel].contiguous(), td, tab, KV_past[sel].contiguous(), bkv, S)
        assert torch.equal(B3, Bn[sel]) and torch.equal(Bh3, Bh[sel]) and torch.equal(KV3, KVn[sel]), mode


# ---------------------------------------------------------------------------------------- D. pooling
@pytest.mark.parametrize("splits", [1, 3])
def test_pool_mean_bounded_grid(dev, splits):
    """ltm_pool_mean_grid with a persistent grid smaller than the unit count (2220 / 6660 units, a multiple of neither
    7 nor 296): the same bits as one CTA per unit, and the fp64 mean."""
    ops, ca = _ops(), _capi()
    Bv, L, T_, e = 37, 60, 32, 768
    k = torch.randn(Bv, L, T_, e, device=dev, generator=_gen(dev, 500 + splits))
    units = Bv * L * splits
    full = ops.pool_mean(k, splits)
    for max_ctas in (7, 296):
        # pool.cu:307  max_ctas > 0 && max_ctas < units -> pool_mean_kernel<F32, LockStep, true>
        assert 0 < max_ctas < units and units % max_ctas != 0
        out = torch.full_like(full, SENT)
        ca.check(ca.lib().ltm_pool_mean_grid(ca.ptr(k), ca.ptr(out), Bv, L, T_, e, splits, max_ctas,
                                             ca.stream_ptr(dev)), "pool_mean_grid")
        assert torch.equal(out, full), max_ctas
    assert _relerr_rows(full.sum(2), k.double().mean(2)) < 1e-6


def test_pool_bins_at_batch_scale(dev):
    """Per-bin pooling of 64 videos x 256 frames == the per-frame pooling summed over each bin's frames in frame order."""
    ops, T = _ops(), _tables()
    Bv, N, L, T_, e = 64, 256, 256, 32, 768
    t = T.rect_tables(L, N, 0.75, 512)
    assert t.xb_rows > 0
    k = torch.randn(Bv, L, T_, e, device=dev, generator=_gen(dev, 510)) * 2
    got = ops.pool_bins(k, t.to(dev)["fbin_ptr"], t.xb_rows)
    x = ops.pool_mean(k, 1)[:, :, 0]
    want = torch.zeros_like(got)
    for r in range(t.xb_rows):
        for f in range(int(t.fbin_ptr[r]), int(t.fbin_ptr[r + 1])):
            want[:, r] += x[:, f]
    assert torch.equal(got, want)


# ---------------------------------------------------------------------------------------- E. sort-based kernels
@pytest.mark.parametrize("ncat", [127, 128])
def test_resample_sorted_peaky_histogram(dev, ncat):
    """300 videos, a histogram with one dominant bin (>= 400 of 512 draws) and both end bins drawn: draws, their sort
    and the gathered positions / basis indices bit-exact."""
    ops, T = _ops(), _tables()
    g = torch.Generator().manual_seed(600 + ncat)
    Bv = 300
    p = torch.rand(Bv, ncat, generator=g) * 0.02 + 1e-4
    peak = torch.randint(1, ncat - 1, (Bv,), generator=g)
    p[torch.arange(Bv), peak] = 6.0 * p.sum(1)
    u = torch.rand(Bv, 512, dtype=torch.float64, generator=g)
    cdf = torch.cumsum(p.double(), 1) / p.double().sum(1, keepdim=True)
    u[:, 0] = 0.5 * cdf[:, 0]                                   # bin 0
    u[:, 1] = 0.5 * (cdf[:, -2] + 1.0)                          # bin ncat - 1
    want = O.inverse_cdf_sample(p, u)
    assert int((want == peak.unsqueeze(1)).sum(1).min()) >= 400
    assert bool((want == 0).any(1).all()) and bool((want == ncat - 1).any(1).all())
    tab = T.rect_tables(8, 256, .75)
    bins, b2b = torch.from_numpy(tab.bins), torch.from_numpy(tab.bin2basis)
    out = ops.resample(p.to(dev), u.to(dev), bins.to(dev), b2b.to(dev), normalize=False, sort=True)
    used = torch.sort(want, -1)[0]
    assert torch.equal(out["b_draw"].cpu().long(), want)
    assert torch.equal(out["b_used"].cpu().long(), used)
    assert torch.equal(out["ts"].cpu(), bins[used])
    assert torch.equal(out["idx"].cpu().long(), b2b.long()[used])


@pytest.mark.parametrize("L", [0, 37])
def test_fold_sample_columns_long_runs(dev, L):
    """Variant G's operator fold with runs longer than 256 columns (crossing the 32-column chunks and the 8-chunk
    unroll), bins 0 and 127 drawn, and N = 100 operator rows (the last CTA has a partial group of 8)."""
    ops = _ops()
    g = torch.Generator().manual_seed(700 + L)
    Bv, N, S, nbins, e = 6, 100, 512, 128, 96
    GT = torch.randn(N, S + L + 4, generator=g).to(dev)                       # row pitch > S + L
    rows = []
    for v, (pk, run) in enumerate([(5, 300), (64, 330), (127, 260), (0, 400), (100, 290), (31, 257)]):
        rest = torch.randint(0, nbins, (S - run - 2,), generator=g)
        rows.append(torch.cat([rest, torch.tensor([0, nbins - 1]), torch.full((run,), pk)]).sort().values)
    b = torch.stack(rows).int()
    start = (b < torch.tensor([5, 64, 127, 0, 100, 31]).int().unsqueeze(1)).sum(1)
    assert bool(((start % 32) != 0).any())                                    # runs start inside a 32-column chunk
    b = b.to(dev)
    A = ops.fold_sample_columns(GT, b, S, L, nbins)
    assert A.shape == (Bv, N, nbins + L)
    onehot = torch.nn.functional.one_hot(b.long(), nbins).double()            # [Bv, S, nbins]
    assert _relerr_rows(A[:, :, :nbins], GT[:, :S].double() @ onehot) < 1e-6
    assert torch.equal(A[:, :, nbins:], GT[:, S:S + L].unsqueeze(0).expand(Bv, -1, -1))
    Rm = torch.randn(Bv, nbins, e, generator=g).double().to(dev)
    k = torch.randn(Bv, L, e, generator=g).double().to(dev)
    xm = torch.gather(Rm, 1, b.long().unsqueeze(-1).expand(-1, -1, e))
    want = GT[:, :S + L].double() @ torch.cat([xm, k], 1)
    assert _relerr_rows(A.double() @ torch.cat([Rm, k], 1), want) < 1e-6
