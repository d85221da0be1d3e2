"""End-to-end parity of the CUDA path (through the C-ABI) with the CPU oracle and the committed reference
goldens over several sequential chunks, plus size-independent properties at the BASELINE shapes."""
import pytest
import torch

from oracle import ltm_oracle as O
from tests.helpers import (TOL_B, TOL_CTX, compare_draws, guard_band, load_golden, make_inputs, make_proj, proj_tensors,
                           relerr)

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev(cuda_device):
    return cuda_device


# Sampled bins are compared with the oracle's own draws from the SAME uniforms, no guard band.  The sampling kernel is
# bit-exact given (p, u) (tests/test_gpu_kernels.py); end to end p carries the rounding of everything upstream, so a
# uniform that sits on a CDF edge can land in the neighbouring bin.  Such flips are counted (and reported by bench.py),
# each one must be a tie within TIE[precision] (`compare_draws`), and the oracle then continues from the bins the CUDA
# path used so that coefficients / contexts of every later chunk are still compared like for like.
TIE = {"tf32": 1e-3, "tf32x3": 2e-5}
FLIPS = {}          # test id -> (flips, draws): printed in the summary line of the session


def _run_rect(dev, N, L, C, Bv, T=32, e=768, Q=32, tau=.75, sticky=True, q_scale=1.0, seed=31, precision="tf32",
              fast_attn=True, proj_operands="fp16", tag=None, **eng_kw):
    from infinite_video_b200.batched import BatchedRectLTM
    key, val = make_proj(seed, e)
    eng = BatchedRectLTM(N, tau, *proj_tensors(key, val), tokens_per_frame=T, sticky=sticky, precision=precision,
                         device=dev, keep_scores=True, fast_attn=fast_attn, proj_operands=proj_operands, **eng_kw)
    orcs = [O.RectLTM(N, tau, *proj_tensors(key, val), tokens_per_frame=T, sticky=sticky, rebuild_tables=False,
                      spacing=eng_kw.get("spacing", "linear")) for _ in range(Bv)]
    ks, qs, us = make_inputs(seed + 1, C, Bv, L * T, e, Q, q_scale)
    worst = dict(B=0.0, ctx=0.0, flips=0, draws=0)
    with torch.no_grad():
        for c in range(C):
            u = us[c]
            upd = c > 0 and sticky
            got = eng.step(ks[c].to(dev), qs[c].to(dev), u.to(dev) if upd else None, new_doc=(c == 0))
            b_got = eng.last["b"].cpu().long() if upd else None
            want = torch.cat([orcs[v].forward(ks[c][v:v + 1], qs[c][v:v + 1], c == 0, u[v:v + 1],
                                              b_override=b_got[v:v + 1] if upd else None) for v in range(Bv)])
            if upd:
                f, d = compare_draws(b_got, torch.cat([o.last["b_own"] for o in orcs]), u,
                                     torch.cat([o.last["p"] for o in orcs]), TIE[precision])
                worst["flips"] += f
                worst["draws"] += d
                assert torch.equal(eng.last["ts"].cpu(), torch.cat([o.last["ts"] for o in orcs]))
                assert torch.equal(eng.last["idx"].cpu().long(), torch.stack([o.last["idx"] for o in orcs]))
            wantB = torch.cat([o.B_past for o in orcs])
            worst["B"] = max(worst["B"], relerr(eng.B_past, wantB))
            worst["ctx"] = max(worst["ctx"], relerr(got, want))
    if tag:
        FLIPS[tag] = (worst["flips"], worst["draws"])
        print(f"[flips] {tag}: {worst['flips']} of {worst['draws']} draws")
    return worst


@pytest.mark.parametrize("name,kw", [
    ("cfg1", dict(N=64, L=8, C=4, Bv=3)),                                   # BASELINE configs[0]
    ("n128", dict(N=128, L=16, C=3, Bv=2, Q=40)),
    ("cfg2", dict(N=256, L=256, C=3, Bv=2)),                                # BASELINE configs[1] (NExT-QA shape)
    ("cfg3", dict(N=64, L=16, C=3, Bv=1, T=196, e=1024, Q=96)),             # BASELINE configs[2] (VideoChat2)
    ("cfg4", dict(N=512, L=32, C=3, Bv=2)),                                 # num_basis=512 stress
    ("peaky", dict(N=64, L=8, C=3, Bv=2, q_scale=8.0, precision="tf32x3")),  # far-from-uniform sticky histogram
    ("peaky_tf32", dict(N=64, L=8, C=3, Bv=2, q_scale=8.0)),
    ("odd", dict(N=64, L=7, C=3, Bv=1)),
    ("nonpow2", dict(N=100, L=30, C=3, Bv=2, tau=.5)),                      # positions that fall in no bin
    ("uniform", dict(N=64, L=8, C=3, Bv=2, sticky=False)),                  # non-sticky re-sampling
    ("log", dict(N=64, L=8, C=3, Bv=2, spacing="log")),                     # N4: log-spaced first-chunk positions
    ("log256", dict(N=256, L=32, C=2, Bv=1, spacing="log")),
    ("cfg2_kv32", dict(N=256, L=256, C=4, Bv=2, kv_dtype="fp32")),          # projected memory on the tf32 grid
    ("cfg1_kv32", dict(N=64, L=8, C=4, Bv=3, kv_dtype="fp32")),             # (the default stores it as fp16)
    ("n128_kv32", dict(N=128, L=16, C=3, Bv=2, Q=40, kv_dtype="fp32")),
    ("cfg4_kv32", dict(N=512, L=32, C=3, Bv=2, kv_dtype="fp32")),
    ("peaky_kv32", dict(N=64, L=8, C=3, Bv=2, q_scale=8.0, kv_dtype="fp32")),
    ("cfg2_p32", dict(N=256, L=256, C=3, Bv=2, proj_operands="fp32")),      # tf32 projection from the fp32 coefficients
    ("cfg2_p32_kv32", dict(N=256, L=64, C=3, Bv=2, proj_operands="fp32", kv_dtype="fp32")),   # the round-1 numerics
    ("cfg4_p32", dict(N=512, L=32, C=3, Bv=2, proj_operands="fp32")),
])
def test_rect_matches_oracle_over_chunks(dev, name, kw):
    w = _run_rect(dev, tag=name, **kw)
    assert w["B"] < 1e-5, w            # the segmented mean is fp32 exact up to summation order
    assert w["ctx"] < TOL_CTX, w       # single-pass TF32 projection, fp32 accumulate
    # ties are rare: at most 1 % of the draws even for the peaky TF32 case (measured rates: bench.py `parity`)
    assert w["flips"] <= 0.01 * max(w["draws"], 1), w


@pytest.mark.parametrize("kw", [dict(N=256, L=32, C=3, Bv=2), dict(N=64, L=8, C=3, Bv=2, Q=96),
                                dict(N=128, L=16, C=3, Bv=3, q_scale=4.0, precision="tf32x3")])
def test_generic_attention_path_still_matches(dev, kw):
    """num_basis 64/128/256 normally take the transposed-key kernels; the generic kernels must agree too."""
    w = _run_rect(dev, fast_attn=False, **kw)
    assert w["B"] < 1e-5 and w["ctx"] < TOL_CTX, w


@pytest.mark.parametrize("N,L,Bv,C,bin_pool", [(64, 8, 2, 48, None), (256, 16, 1, 256, True)])
def test_no_drift_over_a_long_video(dev, N, L, Bv, C, bin_pool):
    """The projected memory K|V is carried from call to call (rounded to fp16 at every store) instead of being
    re-projected from the coefficients: 48 sequential chunks -- and the 256 chunks of a full NExT-QA video
    (BASELINE configs[1]: max_int = 256, num_basis 256) -- against the oracle, which projects afresh every call: the
    context error must stay where it starts (the rounding noise of a carried row is averaged and shrunk by
    g_j * cnt_j < 1 each call), not accumulate."""
    from infinite_video_b200.batched import BatchedRectLTM
    key, val = make_proj(39, 768)
    eng = BatchedRectLTM(N, .75, *proj_tensors(key, val), device=dev, bin_pool=bin_pool)
    assert eng.kv_state and eng.kv_half
    orcs = [O.RectLTM(N, .75, *proj_tensors(key, val), rebuild_tables=False, faithful_quadrature=False)
            for _ in range(Bv)]
    g = torch.Generator().manual_seed(40)
    errs, flips = [], 0
    with torch.no_grad():
        for c in range(C):
            k = torch.randn(Bv, L * 32, 768, generator=g)
            q = torch.randn(Bv, 32, 768, generator=g)
            u = torch.rand(Bv, 512, dtype=torch.float64, generator=g)
            got = eng.step(k.to(dev), q.to(dev), u.to(dev) if c else None, new_doc=(c == 0))
            b_got = eng.last["b"].cpu().long() if c else None
            want = torch.cat([orcs[v].forward(k[v:v + 1], q[v:v + 1], c == 0, u[v:v + 1],
                                              b_override=b_got[v:v + 1] if c else None) for v in range(Bv)])
            if c:
                f, _ = compare_draws(b_got, torch.cat([o.last["b_own"] for o in orcs]), u,
                                     torch.cat([o.last["p"] for o in orcs]), TIE["tf32"])
                flips += f
            assert relerr(eng.B_past, torch.cat([o.B_past for o in orcs])) < 1e-5, c
            errs.append(relerr(got, want))
    assert max(errs) < TOL_CTX, max(errs)
    first, last = sum(errs[1:9]) / 8, sum(errs[-8:]) / 8
    print(f"[drift] ctx error, mean of chunks 1-8: {first:.2e}, of the last 8: {last:.2e}; flips {flips} of {(C - 1) * Bv * 512}")
    assert last < 2 * first + 1e-4
    assert flips <= 0.002 * (C - 1) * Bv * 512


def test_ragged_video_chunk_lengths(dev):
    """A video whose chunks differ in length (the last chunk of a real video is shorter; the reference rebuilds its
    tables for whatever `k.size(1)` it is handed): the memory state carries over between chunk lengths, the carried
    K|V are simply re-projected once after a change of shape.  Also: a change of the query count inside a video is
    refused instead of silently restarting the memory."""
    from infinite_video_b200.batched import BatchedRectLTM
    key, val = make_proj(37, 768)
    N, Bv = 64, 2
    eng = BatchedRectLTM(N, .75, *proj_tensors(key, val), device=dev)
    orcs = [O.RectLTM(N, .75, *proj_tensors(key, val), rebuild_tables=False) for _ in range(Bv)]
    g = torch.Generator().manual_seed(38)
    for c, L in enumerate((16, 16, 8, 8, 5, 16)):
        k = torch.randn(Bv, L * 32, 768, generator=g)
        q = torch.randn(Bv, 32, 768, generator=g)
        u = torch.rand(Bv, 512, dtype=torch.float64, generator=g)
        with torch.no_grad():
            got = eng.step(k.to(dev), q.to(dev), u.to(dev) if c else None, new_doc=(c == 0))
            b_got = eng.last["b"].cpu().long() if c else None
            want = torch.cat([orcs[v].forward(k[v:v + 1], q[v:v + 1], c == 0, u[v:v + 1],
                                              b_override=b_got[v:v + 1] if c else None) for v in range(Bv)])
        if c:
            compare_draws(b_got, torch.cat([o.last["b_own"] for o in orcs]), u, torch.cat([o.last["p"] for o in orcs]),
                          TIE["tf32"])
        assert relerr(eng.B_past, torch.cat([o.B_past for o in orcs])) < 1e-5, (c, L)
        assert relerr(got, want) < TOL_CTX, (c, L)
    with pytest.raises(ValueError):
        eng.step(torch.randn(Bv, 16 * 32, 768, device=dev), torch.randn(Bv, 40, 768, device=dev),
                 torch.rand(Bv, 512, dtype=torch.float64, device=dev))


def test_projected_memory_state_equals_full_projection(dev):
    """kv_state (K|V of the old bins carried from the previous call, only the new-frame rows projected) against the
    engine that projects all N rows every call, over enough chunks for a rounding drift to show: coefficients are
    bit-identical (that path is unchanged), contexts agree well inside the tolerance to the oracle."""
    from infinite_video_b200.batched import BatchedRectLTM
    for N, L, kw in ((256, 64, {}), (512, 32, {}), (64, 8, {}), (256, 64, dict(kv_dtype="fp32")),
                     (256, 64, dict(proj_precision="tf32x3", kv_dtype="fp32")),
                     (256, 32, dict(fast_attn=False, precision="tf32x3"))):
        key, val = make_proj(33, 768)
        a = BatchedRectLTM(N, .75, *proj_tensors(key, val), device=dev, kv_state=True, **kw)
        b = BatchedRectLTM(N, .75, *proj_tensors(key, val), device=dev, kv_state=False, **kw)
        assert a.kv_state and not b.kv_state
        ks, qs, us = make_inputs(34, 10, 3, L * 32, 768, 32)
        worst = 0.0
        for c in range(10):
            k, q, u = ks[c].to(dev), qs[c].to(dev), us[c].to(dev)
            x = a.step(k, q, u if c else None, new_doc=(c == 0))
            y = b.step(k, q, u if c else None, new_doc=(c == 0))
            if c and not torch.equal(a.last["b"], b.last["b"]):
                assert c >= 4, (N, c)          # a draw on a CDF edge went the other way: nothing left to compare
                break
            assert torch.equal(a.B_past, b.B_past), (N, c)
            worst = max(worst, relerr(x, y), relerr(a.last["KV"].float(), b.last["KV"].float()))
        assert worst < (5e-4 if kw.get("precision") != "tf32x3" else 1e-5), (N, kw, worst)


def test_rect_split_tf32_is_fp32_grade(dev):
    w = _run_rect(dev, N=256, L=32, C=3, Bv=2, precision="tf32x3")
    assert w["B"] < 1e-5 and w["ctx"] < 2e-5, w


@pytest.mark.parametrize("bin_pool", [False, True])
@pytest.mark.parametrize("precision", ["tf32", "tf32x3"])
@pytest.mark.parametrize("name", ["gibbs_vl_cfg1.npz", "gibbs_vl_cfg2.npz", "gibbs_vl_peaky.npz",
                                  "gibbs_vc_cfg3.npz", "gibbs_vl_cfg4.npz"])
def test_rect_reproduces_reference_goldens(dev, name, precision, bin_pool):
    """CUDA path vs outputs of the real reference module (tests/golden, generated in the dev container) fed with
    the uniforms the reference itself consumed -- no guard band: the sampled bins must equal the reference's
    (`b`, observed through Categorical.sample by make_golden.py), and with them coefficients and contexts."""
    from infinite_video_b200.batched import BatchedRectLTM
    g = load_golden(name)
    N, L, C, seed, T, e, Q = (int(x) for x in g["meta"])
    key, val = make_proj(seed, e)
    # bin_pool: update chunks pooled per frame (what a one-video engine picks) / per basis bin (the batched headline)
    eng = BatchedRectLTM(N, float(g["tau"]), *proj_tensors(key, val), tokens_per_frame=T, device=dev,
                         precision=precision, bin_pool=bin_pool)
    ks, qs, _ = make_inputs(seed + 1, C, 1, L * T, e, Q, float(g["q_scale"]))
    for c in range(C):
        u = torch.from_numpy(g["u"][c]).to(dev)
        ctx = eng.step(ks[c].to(dev), qs[c].to(dev), u if c else None, new_doc=(c == 0))
        if c:
            b_ref = torch.from_numpy(g["b"][c])
            flips, _ = compare_draws(eng.last["b"], b_ref, g["u"][c], g["p"][c], TIE[precision])
            assert flips == 0, f"{name}/{precision}: {flips} sampled bins differ from the reference's at chunk {c}"
            assert relerr(eng.last["p"], g["p"][c]) < (2e-3 if precision == "tf32" else 2e-5)
        assert relerr(eng.B_past[0, :, :96], g["B_cols"][c]) < TOL_B, f"{name}: B, chunk {c}"
        assert relerr(ctx[0], g["ctx"][c]) < TOL_CTX, f"{name}: ctx, chunk {c}"


def test_cfg4_at_full_size(dev):
    """BASELINE configs[3]: num_basis=512, 64 videos, chunks of 256 frames, sticky re-sampling on every chunk.  The
    CUDA path runs the whole batch; the oracle checks a spread of its videos (a CPU call at this size takes ~1 s)."""
    N, L, Bv, C = 512, 256, 64, 3
    from infinite_video_b200.batched import BatchedRectLTM
    key, val = make_proj(15, 768)
    eng = BatchedRectLTM(N, .75, *proj_tensors(key, val), device=dev)
    check = [0, 21, 42, 63]
    orcs = {v: O.RectLTM(N, .75, *proj_tensors(key, val), rebuild_tables=False, faithful_quadrature=False)
            for v in check}
    g = torch.Generator().manual_seed(16)
    flips = draws = 0
    with torch.no_grad():
        for c in range(C):
            k = torch.randn(Bv, L * 32, 768, generator=g)
            q = torch.randn(Bv, 32, 768, generator=g)
            u = torch.rand(Bv, 512, dtype=torch.float64, generator=g)
            got = eng.step(k.to(dev), q.to(dev), u.to(dev) if c else None, new_doc=(c == 0)).cpu()
            assert torch.isfinite(got).all()
            b_got = eng.last["b"].cpu().long()
            for v in check:
                o = orcs[v]
                want = o.forward(k[v:v + 1], q[v:v + 1], c == 0, u[v:v + 1], b_override=b_got[v:v + 1] if c else None)
                if c:
                    f, d = compare_draws(b_got[v:v + 1], o.last["b_own"], u[v:v + 1], o.last["p"], TIE["tf32"])
                    flips, draws = flips + f, draws + d
                assert relerr(eng.B_past[v], o.B_past[0]) < 1e-5, (c, v)
                assert relerr(got[v], want[0]) < TOL_CTX, (c, v)
    print(f"[flips] cfg4 full size: {flips} of {draws} draws")
    assert flips <= 0.01 * draws


def test_host_entry_point_equals_device_entry_point(dev):
    from infinite_video_b200.batched import BatchedRectLTM
    key, val = make_proj(3, 768)
    a = BatchedRectLTM(64, .75, *proj_tensors(key, val), device=dev)
    b = BatchedRectLTM(64, .75, *proj_tensors(key, val), device=dev)
    ks, qs, us = make_inputs(4, 3, 2, 8 * 32, 768, 32)
    for c in range(3):
        x = a.step(ks[c].to(dev), qs[c].to(dev), us[c].to(dev) if c else None, new_doc=(c == 0))
        y = b.step_host(ks[c].pin_memory(), qs[c].pin_memory(), us[c].pin_memory(), new_doc=(c == 0))
        torch.cuda.synchronize()
        assert torch.equal(x.cpu(), y)


def test_drop_in_module(dev):
    """`LongTermAttention` with the caller's keyword set (Qformer.py:135-158) against the oracle, uniforms drawn
    from torch's global CPU generator exactly like the CPU reference (512 used + 512 discarded per call)."""
    from infinite_video_b200 import LongTermAttention
    from oracle.ref_loader import caller_kwargs
    key, val = make_proj(9, 768)
    key, val = key.to(dev), val.to(dev)
    m = LongTermAttention(**caller_kwargs(64, .75, True, key, val))
    kc, vc = key.cpu(), val.cpu()
    orc = O.RectLTM(64, .75, kc.weight.detach(), kc.bias.detach(), vc.weight.detach(), vc.bias.detach())
    ks, qs, _ = make_inputs(10, 3, 1, 8 * 32, 768, 32)
    for c in range(3):
        m.length = m.target_len = ks[c].shape[1]                 # what the caller does (Qformer.py:218-219)
        torch.manual_seed(400 + c)
        got = m(ks[c].to(dev), qs[c].to(dev), new_doc=(c == 0), layer_n=0).detach()
        nxt = torch.rand(1, dtype=torch.float64)
        torch.manual_seed(400 + c)
        u = torch.rand(1, 512, dtype=torch.float64)
        torch.rand(512, dtype=torch.float64)
        assert c == 0 or nxt.item() == torch.rand(1, dtype=torch.float64).item()      # RNG accounting
        with torch.no_grad():
            want = orc.forward(ks[c], qs[c], c == 0, u)
        assert got.shape == (1, 32, 768) and got.dtype == torch.float32
        assert relerr(m.B_past, orc.B_past) < 1e-5
        assert relerr(got, want) < TOL_CTX
    with pytest.raises(RuntimeError):
        m(ks[0], qs[0], new_doc=True, layer_n=0)                 # CPU tensors: no silent fallback


# ------------------------------------------------------------------------------------------------ variant G
def _gauss_ctx_fp64(B, q, key, val, psi, H=12, d=64):
    """Exact-arithmetic (fp64) evaluation of long_term_attention.py:279-325 from given coefficients B."""
    B, q = B.double().cpu(), q.double().cpu()
    bsz, N, _ = B.shape
    K = (B @ key.weight.double().t() + key.bias.double()).view(bsz, N, H, d).transpose(1, 2)
    V = (B @ val.weight.double().t() + val.bias.double()).view(bsz, N, H, d).transpose(1, 2)
    qh = q.view(bsz, -1, H, d).transpose(1, 2) / (d ** 0.5)
    a = torch.softmax(20 * (qh @ K.transpose(-1, -2)), -1)
    bm, bs = psi.mu[0].double(), psi.sigma[0].double()
    mu = a @ bm
    var = a @ (bm ** 2 + bs ** 2) - mu ** 2
    s = torch.sqrt(bs ** 2 + var.unsqueeze(-1))
    r = torch.exp(-0.5 * ((mu.unsqueeze(-1) - bm) / s) ** 2) / (2 * torch.pi) ** 0.5 / s      # [b,h,q,N]
    return (r @ V).transpose(1, 2).reshape(bsz, -1, H * d)


@pytest.mark.parametrize("N,L,Bv,C", [(64, 8, 2, 3), (256, 256, 1, 3), (256, 64, 2, 2)])
def test_gauss_matches_oracle_with_shared_operators(dev, N, L, Bv, C):
    """B / ctx parity of variant G with the ridge operators injected from the oracle: the reference's fp32
    `.inverse()` of a cond~5e5 system is not a reproducible target (SURVEY.md 0.5), everything downstream is."""
    from infinite_video_b200.batched import BatchedGaussLTM
    key, val = make_proj(41, 768)
    orc = O.GaussLTM(N, .75, *proj_tensors(key, val), rebuild_tables=False)
    eng = BatchedGaussLTM(N, .75, *proj_tensors(key, val), device=dev)
    tb = orc.tables(L)
    eng.set_operators(L, G0=tb["G0"], G_inf=tb["G_inf"])
    ks, qs, us = make_inputs(42, C, Bv, L, 768, 32)
    with torch.no_grad():
        for c in range(C):
            # no guard band: the uniforms go in as drawn; the oracle continues with the bins the CUDA path sampled and
            # its own draws are compared with them -- a difference must be a tie on a CDF edge (helpers.compare_draws)
            u = us[c]
            got = eng.step(ks[c].to(dev), qs[c].to(dev), u.to(dev) if c else None, new_doc=(c == 0))
            b_got = eng.last["b"].cpu().long() if c else None
            want = orc.forward(ks[c], qs[c], c == 0, u, b_override=b_got)
            if c > 0:
                flips, _ = compare_draws(b_got, orc.last["b_own"], u, orc.last["p"], 1e-5)
                assert flips <= 2, f"{flips} flipped draws at chunk {c}"
                assert torch.equal(eng.last["ts"].cpu(), orc.last["ts"])
            assert relerr(eng.B_past, orc.B_past) < TOL_B, f"B, chunk {c}"
            # ctx: 1e-3 wherever the reference's own result is well conditioned.  Its variance
            # sigma^2 = E[t^2] - mu^2 (long_term_attention.py:291) is a cancelling subtraction of two ~0.5-sized fp32
            # numbers; when softmax(20 S) is so peaky that sigma^2 drops below 5e-5, four of fp32's seven digits are
            # gone and the reference's own context is several 1e-3 away from exact arithmetic (measured here: reference
            # vs fp64 3.3e-3, CUDA path vs fp64 1.0e-3 at min sigma^2 = 2.5e-5; <= 1.1e-4 to the reference in every other
            # case).  There -- decided by the CONDITIONING of the reference, not by the error -- the CUDA path must be
            # at least as close to exact arithmetic as the reference is, and within 5e-3 of it.
            err = relerr(got, want)
            if float(orc.last["var"].min()) >= 5e-5:
                assert err < TOL_CTX, (c, err)
            else:
                ours = relerr(got, _gauss_ctx_fp64(eng.B_past, qs[c], key, val, tb["psi"]))
                theirs = relerr(want, _gauss_ctx_fp64(orc.B_past, qs[c], key, val, tb["psi"]))
                assert err < 5e-3 and ours <= 1.5 * max(theirs, 1e-4), (c, err, ours, theirs)


@pytest.mark.parametrize("Bv,round1", [(2, False), (64, True)])
def test_gauss_folded_operator_equals_gathered_samples(dev, Bv, round1):
    """Variant G sticky update through the per-video folded operator (default) and through the gathered sample rows:
    same coefficients (two summation orders of one product), same draws, same contexts.  `round1`: the whole round-1
    route on the other side (gathered samples, split-TF32 projection, FMA attention) against today's defaults (folded
    operator, fp16x2 projection, tensor-core attention) at a batch of 64 videos."""
    from infinite_video_b200.batched import BatchedGaussLTM
    key, val = make_proj(43, 768)
    a = BatchedGaussLTM(256, .75, *proj_tensors(key, val), device=dev, fold_samples=True)
    kw = dict(proj_precision="tf32x3", tc_attn=False) if round1 else {}
    b = BatchedGaussLTM(256, .75, *proj_tensors(key, val), device=dev, fold_samples=False, **kw)
    assert a.tc_attn and (not round1 or not b.tc_attn)
    ks, qs, us = make_inputs(44, 3, Bv, 64, 768, 32)
    same = torch.ones(Bv, dtype=torch.bool)
    for c in range(3):
        x = a.step(ks[c].to(dev), qs[c].to(dev), us[c].to(dev) if c else None, new_doc=(c == 0))
        y = b.step(ks[c].to(dev), qs[c].to(dev), us[c].to(dev) if c else None, new_doc=(c == 0))
        if c:
            # the two routes hand slightly different (mu, sd) to the erf histogram: a uniform on a CDF edge may land in
            # the neighbouring bin -- verified to be a tie, and that video is left out from then on
            flips, _ = compare_draws(a.last["b"], b.last["b"], us[c], b.last["p"].cpu(), 1e-5)
            assert flips <= 2, (c, flips)
            same &= (a.last["b"] == b.last["b"]).all(dim=1).cpu()
        assert relerr(a.B_past[same], b.B_past[same]) < 2e-5, c
        assert relerr(x[same], y[same]) < 5e-4, c
    assert int(same.sum()) >= Bv - 2


def test_gauss_device_ridge_end_to_end(dev):
    """With its own fp64 device-solved operators the module must track an fp64-operator oracle."""
    import math
    from infinite_video_b200.batched import BatchedGaussLTM
    N, L, Bv = 64, 8, 2
    key, val = make_proj(43, 768)
    eng = BatchedGaussLTM(N, .75, *proj_tensors(key, val), device=dev)
    # fp64-exact operators for the oracle
    psi = O.GaussBasis(N, [0.005, 0.01])

    def exact(pos, l):
        z = (pos.double().unsqueeze(0) - psi.mu[0].double().unsqueeze(1)) / psi.sigma[0].double().unsqueeze(1)
        F = torch.exp(-0.5 * z * z) / math.sqrt(2 * math.pi) / psi.sigma[0].double().unsqueeze(1)
        G = torch.linalg.solve(F @ F.t() + 0.5 * torch.eye(N, dtype=torch.float64), F).t()
        return G[l // 2:-(l // 2)].float()

    pos_inf, _ = O.update_positions(L, .75)
    orc = O.GaussLTM(N, .75, *proj_tensors(key, val), rebuild_tables=False,
                     tables_override={L: dict(G0=exact(O.first_chunk_positions(L), L), G_inf=exact(pos_inf, 512 + L))})
    ks, qs, us = make_inputs(44, 2, Bv, L, 768, 32)
    with torch.no_grad():
        for c in range(2):
            u = guard_band(us[c], orc.sticky_hist(orc.tables(L))) if c else us[c]
            want = orc.forward(ks[c], qs[c], c == 0, u)
            got = eng.step(ks[c].to(dev), qs[c].to(dev), u.to(dev) if c else None, new_doc=(c == 0))
            assert relerr(eng.B_past, orc.B_past) < TOL_B
            assert relerr(got, want) < TOL_CTX


# ------------------------------------------------------------------------------------------------ properties
def test_full_size_properties(dev):
    """Size-independent checks at the NExT-QA shape (L=256, N=256, 32x768 tokens) with a batch of videos."""
    from infinite_video_b200 import tables
    from infinite_video_b200.batched import BatchedRectLTM
    key, val = make_proj(51, 768)
    N, L, Bv = 256, 256, 8
    g = torch.Generator(device=dev).manual_seed(5)
    k0 = torch.randn(Bv, L * 32, 768, device=dev, generator=g)
    k1 = torch.randn(Bv, L * 32, 768, device=dev, generator=g)
    q = torch.randn(Bv, 32, 768, device=dev, generator=g)
    u = torch.rand(Bv, 512, device=dev, dtype=torch.float64, generator=g)
    eng = BatchedRectLTM(N, .75, *proj_tensors(key, val), device=dev)
    c0 = eng.step(k0, q, None, new_doc=True).clone()
    B0 = eng.B_past.clone()
    c1 = eng.step(k1, q, u, new_doc=False).clone()
    B1 = eng.B_past.clone()
    assert torch.isfinite(c0).all() and torch.isfinite(c1).all()
    # (i) restarting the document reproduces the same bits (state fully reset, kernels deterministic)
    assert torch.equal(eng.step(k0, q, None, new_doc=True), c0)
    assert torch.equal(eng.step(k1, q, u, new_doc=False), c1)
    # (ii) batch invariance: a video consolidated in a smaller batch gives the same bits as inside the big one
    #      (alone, the frame pooling is split over more CTAs to fill the GPU: same value up to summation order)
    half = BatchedRectLTM(N, .75, *proj_tensors(key, val), device=dev)
    h0 = half.step(k0[2:6], q[2:6], None, new_doc=True)
    h1 = half.step(k1[2:6], q[2:6], u[2:6], new_doc=False)
    # (a smaller batch pools with more token-splits per frame to fill the GPU: same value up to summation order; 1e-7
    # differences in B can cross a tf32 rounding boundary of K, V or the attention weights, 2^-12 relative each)
    assert relerr(h0, c0[2:6]) < 1e-4 and relerr(h1, c1[2:6]) < 1e-4
    solo = BatchedRectLTM(N, .75, *proj_tensors(key, val), device=dev)
    s0 = solo.step(k0[3:4], q[3:4], None, new_doc=True)
    s1 = solo.step(k1[3:4], q[3:4], u[3:4], new_doc=False)
    # (a solo video pools with a different split count: 1e-7 differences in B can cross a tf32 rounding boundary of
    # K, V or the attention weights, each worth 2^-12 relative on one element)
    assert relerr(s0[0], c0[3]) < 1e-4 and relerr(s1[0], c1[3]) < 1e-4
    # (iii) linearity of the regression in the chunk: B(2k) == 2 B(k) exactly (power-of-two scaling)
    eng.step(2 * k0, q, None, new_doc=True)
    assert torch.equal(eng.B_past, 2 * B0)
    # (iv) first-chunk coefficients are shrunk bin means: every frame is alone in its bin at L == N
    x = k0.view(Bv, L, 32, 768).mean(2)
    assert relerr(B0, x / 1.5) < 1e-6
    # (v) the last new frame of an update chunk is dropped (its position 1.0 lies in no bin)
    k1b = k1.clone()
    k1b.view(Bv, L, 32, 768)[:, -1] += 100.0
    eng.step(k0, q, None, new_doc=True)
    eng.step(k1b, q, u, new_doc=False)
    assert torch.equal(eng.B_past, B1)
    # (vi) zero queries: S == 0 so r_j == W_j exactly and ctx == sum_j W_j V_j  (W sums to 1 - W_out)
    eng.step(k0, torch.zeros_like(q), None, new_doc=True)
    V = eng.last["V"]
    W = tables.rect_tables(L, N, .75).to(dev)["W"]
    want = torch.einsum("j,vjd->vd", W / (W.sum() + tables.rect_tables(L, N, .75).W_out), V.float())
    got = eng.step(k0, torch.zeros_like(q), None, new_doc=True)
    # (the tensor-core attention rounds the weights W_j and the values to tf32: 2^-12 relative per element)
    assert relerr(got[:, 0], want) < 2e-4 and relerr(got[:, 31], want) < 2e-4


def test_prefetched_pooling_is_bit_identical(dev):
    """Pooling chunk c+1 ahead of time on the side stream (full or bounded grid) must not change a single bit."""
    from infinite_video_b200.batched import BatchedRectLTM
    key, val = make_proj(61, 768)
    a = BatchedRectLTM(256, .75, *proj_tensors(key, val), device=dev)
    b = BatchedRectLTM(256, .75, *proj_tensors(key, val), device=dev)
    b.pool_ctas = 148 * 2
    ks, qs, us = make_inputs(62, 4, 4, 64 * 32, 768, 32)
    ks = [k.to(dev) for k in ks]
    qs = [q.to(dev) for q in qs]
    us = [u.to(dev) for u in us]
    b.prefetch(ks[0], 32)
    for c in range(4):
        x = a.step(ks[c], qs[c], us[c] if c else None, new_doc=(c == 0))
        if c + 1 < 4:
            b.prefetch(ks[c + 1], 32)             # next chunk is pooled while this one is consolidated
        y = b.step(ks[c], qs[c], us[c] if c else None, new_doc=(c == 0))
        assert torch.equal(x, y), f"chunk {c}"
        assert torch.equal(a.B_past, b.B_past)


@pytest.mark.parametrize("N,L,Bv", [(256, 64, 3), (256, 256, 2), (512, 256, 2), (64, 8, 2)])
def test_per_bin_pooling_matches_per_frame_pooling(dev, N, L, Bv):
    """`bin_pool=True` (frames of an update chunk pooled per basis bin, csrc/pool.cu) against `bin_pool=False`: bins
    with frames only are bit-identical, a bin that mixes re-sampled memory and frames adds them in another order
    (1 ulp); through `step`, `prefetch(update=True)` + `step`, `step_overlapped`, and a chunk that was pooled per bin
    but then starts a new document (pooled again per frame)."""
    from infinite_video_b200.batched import BatchedRectLTM
    key, val = make_proj(67, 768)
    mk = lambda bp: BatchedRectLTM(N, .75, *proj_tensors(key, val), device=dev, bin_pool=bp)
    a, b, c, d = mk(False), mk(True), mk(True), mk(True)
    C = 5
    ks, qs, us = make_inputs(68, C, Bv, L * 32, 768, 32)
    ks = [k.to(dev) for k in ks]
    qs = [q.to(dev) for q in qs]
    us = [u.to(dev) for u in us]
    firsts = [True, False, False, True, False]                        # chunk 3 starts a new document
    for i in range(C):
        u = None if firsts[i] else us[i]
        x = a.step(ks[i], qs[i], u, new_doc=firsts[i])
        y = b.step(ks[i], qs[i], u, new_doc=firsts[i])
        if i + 1 < C:
            c.prefetch(ks[i + 1], 32, update=True)                    # wrong guess for chunk 3: pooled again
        z = c.step(ks[i], qs[i], u, new_doc=firsts[i])
        w = d.step_overlapped(ks[i], qs[i], u, new_doc=firsts[i], k_next=ks[i + 1] if i + 1 < C else None,
                              next_new_doc=(i + 1 < C and firsts[i + 1] and i != 2))   # i == 2: wrong hint on purpose
        for other in (b, c, d):
            assert relerr(other.B_past, a.B_past) < 1e-6, i
            assert firsts[i] or torch.equal(other.last["b"], a.last["b"]), i
        assert torch.equal(y, z) and torch.equal(y, w), i
        assert relerr(y, x) < 1e-4, i          # a 1-ulp coefficient can round to the neighbouring fp16 key / value
        if not firsts[i]:
            xa, xb = a.x_past(), b.x_past()                           # the frames are pooled again on demand
            assert torch.equal(xb[:, :, 512:], xa[:, :, 512:]) and relerr(xb, xa) < 1e-6


def test_prefetch_bookkeeping_survives_abandoned_and_interleaved_chunks(dev):
    """Pending prefetches are keyed on tensor identity + version, never on the data pointer: an abandoned prefetch,
    a non-prefetched step in between, a recycled address or an in-place rewrite must not make a step consume stale
    pooled frames (results stay bit-identical to plain `step`)."""
    from infinite_video_b200.batched import BatchedRectLTM
    key, val = make_proj(65, 768)
    a = BatchedRectLTM(64, .75, *proj_tensors(key, val), device=dev)
    b = BatchedRectLTM(64, .75, *proj_tensors(key, val), device=dev)
    ks, qs, us = make_inputs(66, 6, 2, 8 * 32, 768, 32)
    ks = [k.to(dev) for k in ks]
    qs = [q.to(dev) for q in qs]
    us = [u.to(dev) for u in us]

    def both(c, first, **kw):
        x = a.step(ks[c], qs[c], None if first else us[c], new_doc=first)
        y = b.step(ks[c], qs[c], None if first else us[c], new_doc=first, **kw)
        assert torch.equal(x, y), f"chunk {c}"
    # (c) prefetch(A) -> plain step(B) -> prefetch(C) -> step(A) -> step(C): A's pooled frames must survive
    b.prefetch(ks[1], 32)
    both(0, True)
    b.prefetch(ks[2], 32)
    both(1, False)
    both(2, False)
    # (a) an abandoned prefetch, then a NEW tensor that recycles its address and shape
    junk = torch.randn_like(ks[3])
    b.prefetch(junk, 32)
    addr = junk.data_ptr()
    del junk
    fresh = ks[3].clone()
    if fresh.data_ptr() == addr:                       # the caching allocator usually hands the block back
        x = a.step(ks[3], qs[3], us[3])
        y = b.step(fresh, qs[3], us[3])
        assert torch.equal(x, y)
    else:
        both(3, False)
    # in-place rewrite behind an unchanged pointer: the version counter invalidates the prefetch
    buf = ks[4].clone()
    b.prefetch(buf, 32)
    buf.copy_(ks[5])
    x = a.step(ks[5], qs[4], us[4])
    y = b.step(buf, qs[4], us[4])
    assert torch.equal(x, y)
    # (b) more prefetches than buffers: the oldest is evicted, nothing raises, and reset() forgets them all
    for c in range(4):
        b.prefetch(ks[c], 32)
    assert len(b._pref) == 2
    b.reset(); a.reset()
    assert not b._pref
    both(0, True)
    with pytest.raises(ValueError):
        b.prefetch(ks[0].transpose(1, 2), 32)          # a copy made by .contiguous() could never be matched later


def test_overlapped_step_is_bit_identical(dev):
    """`step_overlapped` (one library call: this chunk's kernels on a high-priority stream, the next chunk's frame
    pooling on a side stream, joined into the caller's stream) == `step`, bit for bit, over a whole stream of chunks,
    including a second video that starts without a pending prefetch."""
    from infinite_video_b200.batched import BatchedRectLTM
    key, val = make_proj(63, 768)
    a = BatchedRectLTM(256, .75, *proj_tensors(key, val), device=dev)
    b = BatchedRectLTM(256, .75, *proj_tensors(key, val), device=dev)
    ks, qs, us = make_inputs(64, 5, 3, 64 * 32, 768, 32)
    ks = [k.to(dev) for k in ks]
    qs = [q.to(dev) for q in qs]
    us = [u.to(dev) for u in us]
    for rep in range(2):
        for c in range(5):
            x = a.step(ks[c], qs[c], us[c] if c else None, new_doc=(c == 0))
            nxt = ks[c + 1] if c + 1 < 5 else None
            y = b.step_overlapped(ks[c], qs[c], us[c] if c else None, new_doc=(c == 0), k_next=nxt)
            assert torch.equal(x, y), f"rep {rep} chunk {c}"
            assert torch.equal(a.B_past, b.B_past)
    torch.cuda.synchronize()


def test_headline_batch_overlapped_equals_plain(dev):
    """The bench configuration at size (128 videos x 256 frames, num_basis 256): `step_overlapped` with its defaults --
    update chunks pooled per basis bin, four consolidation rows per CTA, the projection confined to part of the SMs
    beside the pooling -- against plain `step` calls of an engine that pools per frame; and three of the videos against
    the oracle."""
    from infinite_video_b200.batched import BatchedRectLTM
    from infinite_video_b200 import tables as _T
    key, val = make_proj(91, 768)
    N, L, Bv, C = 256, 256, 128, 3
    a = BatchedRectLTM(N, .75, *proj_tensors(key, val), device=dev, bin_pool=False)
    b = BatchedRectLTM(N, .75, *proj_tensors(key, val), device=dev)
    assert b._bin_ok(Bv, L, _T.rect_tables(L, N, .75, 512)) and b.gemm_ctas_overlap > 0
    check = [0, 63, 127]
    orcs = {v: O.RectLTM(N, .75, *proj_tensors(key, val), rebuild_tables=False, faithful_quadrature=False)
            for v in check}
    g = torch.Generator(device=dev).manual_seed(92)
    ks = [torch.randn(Bv, L * 32, 768, device=dev, generator=g) for _ in range(C)]
    qs = [torch.randn(Bv, 32, 768, device=dev, generator=g) for _ in range(C)]
    us = [torch.rand(Bv, 512, dtype=torch.float64, device=dev, generator=g) for _ in range(C)]
    with torch.no_grad():
        for c in range(C):
            x = a.step(ks[c], qs[c], us[c] if c else None, new_doc=(c == 0))
            y = b.step_overlapped(ks[c], qs[c], us[c] if c else None, new_doc=(c == 0),
                                  k_next=ks[c + 1] if c + 1 < C else None)
            assert relerr(b.B_past, a.B_past) < 1e-6, c
            if c:
                assert torch.equal(b.last["b"], a.last["b"]), c
            assert relerr(y, x) < 1e-4, c
            b_got = b.last["b"].cpu().long() if c else None
            for v in check:
                want = orcs[v].forward(ks[c][v:v + 1].cpu(), qs[c][v:v + 1].cpu(), c == 0, us[c][v:v + 1].cpu(),
                                       b_override=b_got[v:v + 1] if c else None)
                if c:
                    compare_draws(b_got[v:v + 1], orcs[v].last["b_own"], us[c][v:v + 1].cpu(), orcs[v].last["p"],
                                  TIE["tf32"])
                assert relerr(b.B_past[v:v + 1], orcs[v].B_past) < TOL_B, (c, v)
                assert relerr(y[v:v + 1], want) < TOL_CTX, (c, v)
    torch.cuda.synchronize()


def test_fp32_projection_operands(dev):
    """`proj_operands="fp32"`: tf32 UMMAs straight from the fp32 coefficients and weights (the default converts both to
    fp16 first).  Same tolerances; the coefficients themselves are fp32 either way."""
    for kw in (dict(N=256, L=64, C=3, Bv=2), dict(N=128, L=16, C=3, Bv=2, Q=40)):
        w = _run_rect(dev, proj_operands="fp32", **kw)
        assert w["B"] < 1e-5 and w["ctx"] < TOL_CTX, w


def test_step_is_cuda_graph_capturable(dev):
    """No host synchronisation / allocation inside a step: a sticky chunk can be captured once and replayed
    (this is how a single-video, launch-bound caller amortises the 5 launches)."""
    from infinite_video_b200.batched import BatchedRectLTM
    key, val = make_proj(71, 768)
    ks, qs, us = make_inputs(72, 4, 1, 32 * 32, 768, 32)
    ks = [k.to(dev) for k in ks]
    qs = [q.to(dev) for q in qs]
    us = [u.to(dev) for u in us]
    ref = BatchedRectLTM(256, .75, *proj_tensors(key, val), device=dev)
    want = [ref.step(ks[c], qs[c], us[c] if c else None, new_doc=(c == 0)).clone() for c in range(4)]

    eng = BatchedRectLTM(256, .75, *proj_tensors(key, val), device=dev)
    k_s, q_s, u_s = ks[0].clone(), qs[0].clone(), us[1].clone()
    eng.step(k_s, q_s, None, new_doc=True)                      # chunk 0 (eager)
    k_s.copy_(ks[1]); q_s.copy_(qs[1])
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):                                 # warm-up of the update path on a side stream
        eng.step(k_s, q_s, u_s, new_doc=False)
    torch.cuda.current_stream().wait_stream(side)
    # rewind the state to "after chunk 0" and capture one update step; two captures alternate the ping-pong
    eng.reset()
    k_s.copy_(ks[0]); q_s.copy_(qs[0])
    eng.step(k_s, q_s, None, new_doc=True)
    a = eng._cur                                                  # buffer that holds B after chunk 0
    graphs, outs = [], []
    for _ in range(2):                                            # B_past ping-pong: one graph per parity
        g = torch.cuda.CUDAGraph()
        k_s.copy_(ks[1]); q_s.copy_(qs[1]); u_s.copy_(us[1])
        with torch.cuda.graph(g):
            out = eng.step(k_s, q_s, u_s, new_doc=False)
        graphs.append(g); outs.append(out)
    # replay from scratch: chunk 0 eager, chunks 1..3 through the graphs
    eng.reset()
    eng._cur = 1 - a                                              # so that chunk 0 lands in the buffer graph 0 reads
    k_s.copy_(ks[0]); q_s.copy_(qs[0])
    assert torch.equal(eng.step(k_s, q_s, None, new_doc=True), want[0])
    for c in range(1, 4):
        k_s.copy_(ks[c]); q_s.copy_(qs[c]); u_s.copy_(us[c])
        i = (c - 1) & 1
        graphs[i].replay()
        assert torch.equal(outs[i], want[c]), f"graph replay differs at chunk {c}"


def test_layers_share_one_pooling_pass(dev):
    """N2: two LTM layers (different projections, same encoder_hidden_states) -- the second layer must reuse the
    pooled frames of the first and still match an instance that pools on its own, bit for bit."""
    from infinite_video_b200 import LongTermAttention, ops
    from oracle.ref_loader import caller_kwargs
    layers, solo = [], []
    for seed in (81, 82):
        key, val = make_proj(seed, 768)
        key, val = key.to(dev), val.to(dev)
        layers.append(LongTermAttention(**caller_kwargs(64, .75, True, key, val)))
        solo.append(LongTermAttention(**caller_kwargs(64, .75, True, key, val), share_pooling=False))
    ks, qs, us = make_inputs(83, 3, 1, 8 * 32, 768, 32)
    calls = {"n": 0}
    real = ops.pool_mean

    def counting(*a, **kw):
        calls["n"] += 1
        return real(*a, **kw)
    ops.pool_mean = counting
    try:
        for c in range(3):
            k = ks[c].to(dev)
            for li in range(2):
                got = layers[li](k, qs[c].to(dev), new_doc=(c == 0), layer_n=li, u=us[c])
                want = solo[li](k, qs[c].to(dev), new_doc=(c == 0), layer_n=li, u=us[c])
                assert torch.equal(got, want), (c, li)
    finally:
        ops.pool_mean = real
    assert calls["n"] == 3          # one pooling pass per chunk for the two sharing layers (solo ones pool in-step)


def test_consolidate_video_chunk_loop(dev):
    """N2, second half: the model-level chunk loop -- all LTM layers of a Q-former, a batch of videos, the frames of
    each chunk pooled once (ahead of time, on a side stream) and shared by the layers -- gives the same bits as one
    engine per layer stepped on its own, with C pooling passes instead of layers x C."""
    from infinite_video_b200 import ops
    from infinite_video_b200.batched import BatchedRectLTM
    from infinite_video_b200.video import consolidate_video
    nl, C, Bv, L = 3, 4, 3, 16
    layers = [BatchedRectLTM(64, .75, *proj_tensors(*make_proj(70 + i, 768)), device=dev) for i in range(nl)]
    solo = [BatchedRectLTM(64, .75, *proj_tensors(*make_proj(70 + i, 768)), device=dev) for i in range(nl)]
    ks, _, _ = make_inputs(75, C, Bv, L * 32, 768, 32)
    ks = [k.to(dev) for k in ks]
    g = torch.Generator().manual_seed(76)
    qs = [[torch.randn(Bv, 32, 768, generator=g).to(dev) for _ in range(C)] for _ in range(nl)]
    us = [[torch.rand(Bv, 512, dtype=torch.float64, generator=g).to(dev) for _ in range(C)] for _ in range(nl)]
    calls = {"n": 0}
    real = ops.pool_mean

    def counting(*a, **kw):
        calls["n"] += 1
        return real(*a, **kw)
    ops.pool_mean = counting
    try:
        got = consolidate_video(layers, ks, qs, us)
    finally:
        ops.pool_mean = real
    assert calls["n"] == C
    for li in range(nl):
        for c in range(C):
            want = solo[li].step(ks[c], qs[li][c], us[li][c] if c else None, new_doc=(c == 0))
            assert torch.equal(got[li][c], want), (li, c)
    # running mean over the chunks (what the eval scripts keep), queries produced layer by layer through a callable
    mean = consolidate_video(layers, ks, lambda li, c, prev: qs[li][c], us, reduce="mean")
    for li in range(nl):
        assert relerr(mean[li], torch.stack(got[li]).mean(0)) < 1e-6


def test_density_side_output(dev):
    """N3: `output_density=True` reproduces the alphas tensor of the Video-LLaMA copy (gibbs:320-343)."""
    from infinite_video_b200 import LongTermAttention
    from oracle.ref_loader import caller_kwargs
    for N, L in ((64, 8), (256, 32)):
        key, val = make_proj(91, 768)
        kd, vd = make_proj(91, 768)
        m = LongTermAttention(**caller_kwargs(N, .75, True, kd.to(dev), vd.to(dev)), output_density=True)
        orc = O.RectLTM(N, .75, *proj_tensors(key, val), rebuild_tables=False)
        ks, qs, us = make_inputs(92, 2, 1, L * 32, 768, 32, q_scale=3.0)
        with torch.no_grad():
            for c in range(2):
                m(ks[c].to(dev), qs[c].to(dev), new_doc=(c == 0), layer_n=0, u=us[c])
                orc.forward(ks[c], qs[c], c == 0, us[c])
                want = O.rect_density_alphas(orc, orc.tables(L))
                assert m.alphas.shape == (32, 1, 12, 768)
                assert relerr(m.alphas, want) < 1e-3
                assert abs(float(m.alphas[3, 0, 5].sum()) - 1.0) < 1e-5


def test_dump_hook_and_x_past(dev, tmp_path):
    """Boundary leftovers of the Video-LLaMA copy: `dump_path` writes the pickle relevant_frames.py:11-12 reads
    (gibbs:344-345: a CPU tensor [Q,B,H,768]), and `x_past` is the regression input the reference keeps (:221)."""
    import pickle
    from infinite_video_b200 import LongTermAttention
    from oracle.ref_loader import caller_kwargs
    key, val = make_proj(97, 768)
    kd, vd = make_proj(97, 768)
    path = str(tmp_path / "alphas_uniform")
    m = LongTermAttention(**caller_kwargs(64, .75, True, kd.to(dev), vd.to(dev)), dump_path=path)
    orc = O.RectLTM(64, .75, *proj_tensors(key, val), rebuild_tables=False)
    ks, qs, us = make_inputs(98, 3, 1, 8 * 32, 768, 32)
    assert m.x_past is None
    with torch.no_grad():
        for c in range(3):
            m(ks[c].to(dev), qs[c].to(dev), new_doc=(c == 0), layer_n=0, u=us[c])
            orc.forward(ks[c], qs[c], c == 0, us[c])
            with open(path, "rb") as f:
                dumped = pickle.load(f)
            assert not dumped.is_cuda and dumped.shape == (32, 1, 12, 768)
            assert torch.equal(dumped, m.alphas.cpu())
            assert relerr(dumped, O.rect_density_alphas(orc, orc.tables(8))) < 1e-3
            assert m.x_past.shape == orc.x_past.shape
            assert relerr(m.x_past, orc.x_past) < 1e-5, f"x_past, chunk {c}"
    m.x_past = None
    with pytest.raises(AttributeError):
        m.x_past = torch.zeros(1)


def test_gauss_kl_regularizer_and_per_video_new_doc(dev):
    """N4 / boundary leftovers of variant G: `(ctx, kl_reg)` when kl_regularizer is on (gauss:296-304,389-390), and
    per-video new_doc flags in the batched engine (a video may start while others continue)."""
    from infinite_video_b200 import LongTermAttention
    from infinite_video_b200.batched import BatchedGaussLTM
    from oracle.ref_loader import caller_kwargs
    N, L = 64, 8
    key, val = make_proj(45, 768)
    kd, vd = make_proj(45, 768)
    for mu_0 in (0.5, -1.0):
        kw = caller_kwargs(N, .75, True, kd.to(dev), vd.to(dev), sigmas=[0.005, 0.01])
        kw.update(kl_regularizer=True, sigma_0=0.3, mu_0=mu_0)
        m = LongTermAttention(**kw, variant="gaussian")
        orc = O.GaussLTM(N, .75, *proj_tensors(key, val), rebuild_tables=False, kl_regularizer=True, sigma_0=0.3,
                         mu_0=mu_0)
        m._get_engine(dev).set_operators(L, G0=orc.tables(L)["G0"], G_inf=orc.tables(L)["G_inf"])
        ks, qs, us = make_inputs(46, 2, 2, L, 768, 32)
        with torch.no_grad():
            for c in range(2):
                u = guard_band(us[c], orc.sticky_hist(orc.tables(L))) if c else us[c]
                ctx, kl = m(ks[c].to(dev), qs[c].to(dev), new_doc=(c == 0), layer_n=0, u=u)
                want = orc.forward(ks[c], qs[c], c == 0, u)
                assert relerr(ctx, want) < 5e-3
                assert kl.shape == orc.kl_reg.shape and relerr(kl, orc.kl_reg) < 2e-3, (mu_0, c)
    # per-video flags: video 1 restarts at chunk 1 while video 0 continues
    eng = BatchedGaussLTM(N, .75, *proj_tensors(key, val), device=dev)
    orcs = [O.GaussLTM(N, .75, *proj_tensors(key, val), rebuild_tables=False) for _ in range(2)]
    tb = orcs[0].tables(L)
    eng.set_operators(L, G0=tb["G0"], G_inf=tb["G_inf"])
    ks, qs, us = make_inputs(47, 3, 2, L, 768, 32)
    flags = [[True, True], [False, True], [False, False]]
    with torch.no_grad():
        for c in range(3):
            u = us[c].clone()
            for v in range(2):
                if not flags[c][v]:
                    u[v:v + 1] = guard_band(u[v:v + 1], orcs[v].sticky_hist(tb))
            got = eng.step(ks[c].to(dev), qs[c].to(dev), u.to(dev), new_doc=flags[c])
            for v in range(2):
                want = orcs[v].forward(ks[c][v:v + 1], qs[c][v:v + 1], flags[c][v], u[v:v + 1])
                assert relerr(eng.B_past[v], orcs[v].B_past[0]) < TOL_B, (c, v)
                assert relerr(got[v], want[0]) < 5e-3, (c, v)


def test_fp16_chunk_through_the_drop_in(dev):
    """VideoChat2 flavour under fp16 autocast: k and q arrive as fp16; the module pools the 16-bit chunk directly
    and must equal the fp32 oracle evaluated on the up-cast inputs; the output comes back in q's dtype."""
    from infinite_video_b200 import LongTermAttention
    from oracle.ref_loader import caller_kwargs
    key, val = make_proj(95, 1024)
    kd, vd = make_proj(95, 1024)
    m = LongTermAttention(**caller_kwargs(64, .75, True, kd.to(dev), vd.to(dev)), tokens_per_frame=196)
    orc = O.RectLTM(64, .75, *proj_tensors(key, val), tokens_per_frame=196, rebuild_tables=False)
    ks, qs, us = make_inputs(96, 2, 1, 16 * 196, 1024, 96)
    with torch.no_grad():
        for c in range(2):
            k16, q16 = ks[c].half(), qs[c].half()
            got = m(k16.to(dev), q16.to(dev), new_doc=(c == 0), layer_n=0, u=us[c])
            want = orc.forward(k16.float(), q16.float(), c == 0, us[c])
            assert got.dtype == torch.float16 and got.shape == (1, 96, 768)
            assert relerr(m.B_past, orc.B_past) < 1e-5
            assert relerr(got.float(), want) < 2e-3          # output rounded to fp16 (2^-11) on top of TOL_CTX


# Video-LLaMA: T = 32 tokens per frame, e = D = 768, Q = 32;  VideoChat2 (BASELINE cfg3): T = 196, e = 1024, Q = 96
CALLER_SHAPES = {"videollama": (32, 768, 32), "videochat2": (196, 1024, 96)}
CALLER_MASKS = ("none", "last40", "every_third_frame", "one_frame_left", "all")


def _caller_mask(B, L, T, c):
    """HF's extended encoder mask [B,1,1,LT]: a different masking pattern per video and chunk, -10000 on even chunks
    and finfo(float32).min on odd ones."""
    value = -10000.0 if c % 2 == 0 else torch.finfo(torch.float32).min
    m = torch.zeros(B, L, T)
    for v in range(B):
        kind = CALLER_MASKS[(v + 2 * c) % len(CALLER_MASKS)]
        if kind == "last40":
            m[v].view(-1)[int(round(.6 * L * T)):] = value
        elif kind == "every_third_frame":
            m[v, ::3] = value
        elif kind == "one_frame_left":
            m[v] = value
            m[v, L // 2] = 0.0
        elif kind == "all":
            m[v] = value
    return m.view(B, 1, 1, L * T)


@pytest.mark.parametrize("operands", ["fp16", "fp32"])
@pytest.mark.parametrize("mask", [False, True], ids=["nomask", "mask"])
@pytest.mark.parametrize("shape,alpha,N,L,B", [("videollama", 0.5, 64, 8, 2), ("videollama", 0.9, 256, 64, 1),
                                               ("videollama", 0.7, 256, 256, 2), ("videochat2", 0.5, 64, 16, 2)])
def test_caller_cross_attention_with_ltm_blend_on_gpu(dev, shape, alpha, N, L, B, mask, operands):
    """N1: short-term softmax attention over the chunk + (1-alpha) LTM, against the oracle of the caller
    (bit-identical to the real BertSelfAttention, tests/test_oracle_vs_reference.py), with and without an encoder
    mask."""
    from infinite_video_b200.cross_attention import CrossAttentionLTM
    T, e, Q = CALLER_SHAPES[shape]
    torch.manual_seed(21)
    lq, lk, lv = torch.nn.Linear(768, 768), torch.nn.Linear(e, 768), torch.nn.Linear(e, 768)
    orcs = [O.CrossAttentionLTM(N, .75, alpha, lq.weight.detach(), lq.bias.detach(), lk.weight.detach(),
                                lk.bias.detach(), lv.weight.detach(), lv.bias.detach(), tokens_per_frame=T,
                                rebuild_tables=False)
            for _ in range(B)]
    import copy
    m = CrossAttentionLTM(copy.deepcopy(lq).to(dev), copy.deepcopy(lk).to(dev), copy.deepcopy(lv).to(dev), alpha, N,
                          .75, tokens_per_frame=T, operands=operands)
    g = torch.Generator().manual_seed(22)
    with torch.no_grad():
        for c in range(3):
            hidden = torch.randn(B, Q, 768, generator=g)
            enc = torch.randn(B, L * T, e, generator=g)
            u = torch.rand(B, 512, dtype=torch.float64, generator=g)
            am = _caller_mask(B, L, T, c) if mask else None
            got = m(hidden.to(dev), enc.to(dev), new_video=(c == 0), layer=0, u=u,
                    encoder_attention_mask=None if am is None else am.to(dev))
            b_got = m.long_term_attention._engine.last["b"].cpu().long() if c else None
            want = torch.cat([orcs[v].forward(hidden[v:v + 1], enc[v:v + 1], c == 0, u[v:v + 1],
                                              mask=None if am is None else am[v:v + 1],
                                              b_override=b_got[v:v + 1] if c else None) for v in range(B)])
            if c:
                compare_draws(b_got, torch.cat([o.ltm.last["b_own"] for o in orcs]), u,
                              torch.cat([o.ltm.last["p"] for o in orcs]), TIE["tf32"])
            stm = m.short_term(torch.nn.functional.linear(hidden, lq.weight, lq.bias).to(dev), enc.to(dev),
                               None if am is None else am.to(dev))
            assert relerr(stm, torch.cat([o.last_stm for o in orcs])) < TOL_CTX, f"short-term, chunk {c}"
            assert relerr(got, want) < TOL_CTX, f"blend, chunk {c}"


def test_caller_layers_share_the_pooling_and_fp16_pass(dev):
    """Two cross-attention layers of a Q-former receive the same chunk: the pass that pools its frames and writes its
    fp16 copy runs once per chunk (the second layer finds both in the shared slot), and each layer equals a module that
    works alone."""
    import copy
    from infinite_video_b200 import LongTermAttention, ops
    from infinite_video_b200.cross_attention import CrossAttentionLTM
    torch.manual_seed(31)
    mods, solo = [], []
    for i in range(2):
        lin = [torch.nn.Linear(768, 768).to(dev) for _ in range(3)]
        mods.append(CrossAttentionLTM(*lin, 0.5, 64, .75))
        solo.append(CrossAttentionLTM(*copy.deepcopy(lin), 0.5, 64, .75))
    calls = {"n": 0}
    real = ops.pool_mean_convert

    def counting(*a, **kw):
        calls["n"] += 1
        return real(*a, **kw)
    g = torch.Generator().manual_seed(32)
    outs = []
    ops.pool_mean_convert = counting
    try:
        for c in range(3):
            enc = torch.randn(2, 8 * 32, 768, generator=g).to(dev)
            hs = [torch.randn(2, 32, 768, generator=g).to(dev) for _ in range(2)]
            u = torch.rand(2, 512, dtype=torch.float64, generator=g)
            outs.append((enc, hs, u, [mods[i](hs[i], enc, new_video=(c == 0), layer=i, u=u) for i in range(2)]))
    finally:
        ops.pool_mean_convert = real
    assert calls["n"] == 3
    for c, (enc, hs, u, got) in enumerate(outs):
        for i in range(2):
            LongTermAttention._shared_pool.update(key=None, x=None, k16=None)       # the solo module shares nothing
            want = solo[i](hs[i], enc, new_video=(c == 0), layer=i, u=u)
            assert torch.equal(got[i], want), (c, i)


def test_import_swap_through_the_real_qformer(dev, tmp_path):
    """SURVEY 7.2 step 2: the UNMODIFIED `Qformer.BertSelfAttention` (baseline/_ref on the GPU box, oracle/install_ref.py)
    with its one import line (Qformer.py:50) resolved to `infinite_video_b200` instead of the reference module: two
    cross-attention layers, alpha = 0.5, three chunks, against the same caller running the real reference LTM on the
    CPU.  Uniforms come from torch's global CPU generator in both (same seed before every call)."""
    import copy
    import os
    import infinite_video_b200
    from oracle import ref_loader as RL
    if not RL.reference_available():
        pytest.skip("reference files absent (neither /root/reference nor baseline/_ref)")
    Qref = RL.load_qformer_vl()
    Qswap = RL.load_qformer_vl(ltm_module=infinite_video_b200, pkg="_swap_vl")
    assert Qswap.LongTermAttention is infinite_video_b200.LongTermAttention
    cfg = RL.bert_config(64, 0.75, 0.5)
    torch.manual_seed(11)
    ref_layers = [Qref.BertSelfAttention(cfg, is_cross_attention=True).eval() for _ in range(2)]
    swap_layers = []
    for r in ref_layers:
        m = Qswap.BertSelfAttention(cfg, is_cross_attention=True).eval()
        m.load_state_dict(copy.deepcopy(r.state_dict()), strict=False)
        swap_layers.append(m.to(dev))
        assert isinstance(m.long_term_attention, infinite_video_b200.LongTermAttention)
    g = torch.Generator().manual_seed(12)
    cwd = os.getcwd()
    os.chdir(tmp_path)                       # the reference LTM pickles ./alphas_uniform on every call
    try:
        with torch.no_grad():
            for c in range(3):
                enc = torch.randn(1, 8 * 32, 768, generator=g)
                enc_d = enc.to(dev)
                for li in range(2):
                    hidden = torch.randn(1, 32, 768, generator=g)
                    torch.manual_seed(700 + 10 * c + li)
                    want = ref_layers[li](hidden, position_embedding_ext=torch.zeros(1), layer=li,
                                          encoder_hidden_states=enc, new_video=(c == 0))[0]
                    torch.manual_seed(700 + 10 * c + li)
                    got = swap_layers[li](hidden.to(dev), position_embedding_ext=torch.zeros(1, device=dev), layer=li,
                                          encoder_hidden_states=enc_d, new_video=(c == 0))[0]
                    assert got.is_cuda and got.shape == want.shape
                    assert relerr(got, want) < TOL_CTX, (c, li)
                    assert relerr(swap_layers[li].long_term_attention.B_past,
                                  ref_layers[li].long_term_attention.B_past) < 1e-5, (c, li)
    finally:
        os.chdir(cwd)
