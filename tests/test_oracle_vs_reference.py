"""Pins the clean-room oracle against the UNMODIFIED reference modules.  The reference is not part of this
repository: the tests that run it skip where it is not installed (oracle/install_ref.py), and there the committed
reference outputs carry the pin (tests/test_golden.py, and the known answers of test_kat_from_survey)."""
import os
import tempfile

import pytest
import torch
import torch.nn as nn

from oracle import ltm_oracle as O
from oracle import ref_loader as RL
from tests.helpers import make_inputs, make_proj, proj_tensors

needs_reference = pytest.mark.skipif(not RL.reference_available(), reason="reference modules not installed")


@needs_reference
@pytest.mark.parametrize("flavour,N,L,C,tau,sticky", [
    ("vl", 64, 8, 4, 0.75, True),        # BASELINE cfg1
    ("vl", 256, 256, 2, 0.75, True),     # BASELINE cfg2 shape
    ("vl", 64, 7, 3, 0.75, True),        # odd chunk length
    ("vl", 100, 30, 3, 0.5, True),       # non power-of-two N: positions that fall in no bin
    ("vl", 64, 8, 3, 0.75, False),       # uniform (non-sticky) re-sampling
    ("vc", 64, 16, 2, 0.75, True),       # BASELINE cfg3 shape (14x14 tokens, width 1024)
])
def test_rect_oracle_is_bit_identical(flavour, N, L, C, tau, sticky, tmp_path):
    T, e, Q = (32, 768, 32) if flavour == "vl" else (196, 1024, 96)
    mod = RL.load_gibbs_vl() if flavour == "vl" else RL.load_gibbs_vc()
    key, val = make_proj(3, e)
    ref = mod.LongTermAttention(**RL.caller_kwargs(N, tau, sticky, key, val))
    orc = O.RectLTM(N, tau, *proj_tensors(key, val), tokens_per_frame=T, sticky=sticky)
    ks, qs, _ = make_inputs(4, C, 1, L * T, e, Q)
    cwd = os.getcwd()
    os.chdir(tmp_path)
    try:
        with torch.no_grad():
            for c in range(C):
                torch.manual_seed(100 + c)
                want = ref(ks[c], qs[c], new_doc=(c == 0), layer_n=0)
                torch.manual_seed(100 + c)
                u = torch.rand(1, 512, dtype=torch.float64)
                got = orc.forward(ks[c], qs[c], c == 0, u)
                assert torch.equal(orc.B_past, ref.B_past), f"B differs at chunk {c}"
                if N == 100:
                    # torch.trapz over the reference's permuted (strided) integrand reduces in a different
                    # order than over a contiguous one for this N: 1 ulp (observed 8.6e-8 relative)
                    assert float((got - want).abs().max() / want.abs().max()) < 2e-7
                else:
                    assert torch.equal(got, want), f"ctx differs at chunk {c}"
    finally:
        os.chdir(cwd)


@needs_reference
@pytest.mark.parametrize("N,L,C,Bv", [(64, 8, 4, 1), (256, 256, 2, 1), (64, 8, 3, 3)])
def test_gauss_oracle_is_bit_identical(N, L, C, Bv):
    mod = RL.load_gaussian_vl()
    key, val = make_proj(5, 768)
    ref = mod.LongTermAttention(**RL.caller_kwargs(N, 0.75, True, key, val, sigmas=[0.005, 0.01]))
    ref.device = "cpu"                                   # never updated upstream (long_term_attention.py:32)
    orc = O.GaussLTM(N, 0.75, *proj_tensors(key, val))
    ks, qs, _ = make_inputs(6, C, Bv, L, 768, 32)
    with torch.no_grad():
        for c in range(C):
            ref.length = ref.target_len = L              # the caller does this (Qformer.py:218-219)
            torch.manual_seed(200 + c)
            want = ref(ks[c], qs[c], new_doc=(c == 0), layer_n=0)
            torch.manual_seed(200 + c)
            nn.Linear(N, 1, bias=False); nn.Linear(N, 1, bias=False)   # throw-away inits consume RNG (:92-95)
            u = torch.rand(Bv, 512, dtype=torch.float64)
            got = orc.forward(ks[c], qs[c], c == 0, u)
            assert torch.equal(orc.B_past, ref.B_past), f"B differs at chunk {c}"
            assert torch.equal(got, want), f"ctx differs at chunk {c}"


@needs_reference
@pytest.mark.parametrize("N,L", [(64, 8), (256, 32), (64, 7)])
def test_rect_oracle_log_spacing_and_x_past(N, L, tmp_path):
    """N4: `spacing='log'` (a plain attribute upstream, gibbs:64,114-127) and the `x_past` state (:221)."""
    mod = RL.load_gibbs_vl()
    key, val = make_proj(8, 768)
    ref = mod.LongTermAttention(**RL.caller_kwargs(N, 0.75, True, key, val))
    ref.spacing = "log"
    orc = O.RectLTM(N, 0.75, *proj_tensors(key, val), spacing="log")
    ks, qs, _ = make_inputs(9, 3, 1, L * 32, 768, 32)
    cwd = os.getcwd()
    os.chdir(tmp_path)
    try:
        with torch.no_grad():
            for c in range(3):
                torch.manual_seed(300 + c)
                want = ref(ks[c], qs[c], new_doc=(c == 0), layer_n=0)
                torch.manual_seed(300 + c)
                u = torch.rand(1, 512, dtype=torch.float64)
                got = orc.forward(ks[c], qs[c], c == 0, u)
                assert torch.equal(orc.B_past, ref.B_past) and torch.equal(got, want), f"chunk {c}"
                assert torch.equal(orc.x_past, ref.x_past), f"x_past, chunk {c}"
    finally:
        os.chdir(cwd)


@needs_reference
@pytest.mark.parametrize("mu_0", [0.5, -1.0])
def test_gauss_oracle_kl_regularizer(mu_0):
    """N4: kl_regularizer (long_term_attention.py:296-304,389-390), both branches of its `mu_0 > 0` test."""
    N, L = 64, 8
    mod = RL.load_gaussian_vl()
    key, val = make_proj(5, 768)
    kw = RL.caller_kwargs(N, 0.75, True, key, val, sigmas=[0.005, 0.01])
    kw.update(kl_regularizer=True, sigma_0=0.3, mu_0=mu_0)
    ref = mod.LongTermAttention(**kw)
    ref.device = "cpu"
    orc = O.GaussLTM(N, 0.75, *proj_tensors(key, val), kl_regularizer=True, sigma_0=0.3, mu_0=mu_0)
    ks, qs, _ = make_inputs(6, 2, 2, L, 768, 32)
    with torch.no_grad():
        for c in range(2):
            ref.length = ref.target_len = L
            torch.manual_seed(200 + c)
            want, kl = ref(ks[c], qs[c], new_doc=(c == 0), layer_n=0)
            torch.manual_seed(200 + c)
            nn.Linear(N, 1, bias=False); nn.Linear(N, 1, bias=False)
            u = torch.rand(2, 512, dtype=torch.float64)
            got = orc.forward(ks[c], qs[c], c == 0, u)
            assert torch.equal(got, want) and torch.equal(orc.kl_reg, kl), f"chunk {c}"


def test_kat_from_survey():
    """Known-answer recipe recorded in SURVEY.md section 8c: what the reference computed for a seeded run.  The
    oracle must reproduce it when fed the uniforms the reference draws from the global generator (512 used + 512
    discarded per update call); the reference itself is run too where it is installed."""
    want_ctx = [0.0188084431, 0.0188654512, 0.0189450830, 0.0187147614]     # ctx.abs().mean() per call
    want_B = [0.0118673714, 0.0171778575, 0.0180101022, 0.0171232764]       # B_past.abs().mean() per call
    want_bins = [109, 60, 115, 79, 76, 61, 26, 68, 118, 36]                 # first 10 bins sampled on call 1

    def oracle_run():
        orc = O.RectLTM(64, 0.75, *proj_tensors(key, val))
        for c in range(4):
            k = torch.randn(1, 8 * 32, 768)
            q = torch.randn(1, 32, 768)
            u = None
            if c:
                u = torch.rand(1, 512, dtype=torch.float64)
                torch.rand(512, dtype=torch.float64)
            ctx = orc.forward(k, q, c == 0, u)
            if c == 1:
                assert orc.last["b"][0, :10].tolist() == want_bins
            yield ctx, orc.B_past

    def reference_run():
        m = RL.load_gibbs_vl().LongTermAttention(**RL.caller_kwargs(64, 0.75, True, key, val))
        cwd = os.getcwd()
        os.chdir(tempfile.mkdtemp())
        try:
            for c in range(4):
                k = torch.randn(1, 8 * 32, 768)
                q = torch.randn(1, 32, 768)
                yield m(k, q, new_doc=(c == 0), layer_n=0), m.B_past
        finally:
            os.chdir(cwd)

    runs = [oracle_run] + ([reference_run] if RL.reference_available() else [])
    for run in runs:
        torch.manual_seed(0)
        key = nn.Linear(768, 768)
        val = nn.Linear(768, 768)
        with torch.no_grad():
            for c, (ctx, B) in enumerate(run()):
                assert abs(ctx.abs().mean().item() - want_ctx[c]) < 1e-8, (run.__name__, c)
                assert abs(B.abs().mean().item() - want_B[c]) < 1e-8, (run.__name__, c)


@needs_reference
def test_density_side_output_matches_the_pickle(tmp_path):
    """N3: the oracle's restatement of the density dump equals what the Video-LLaMA copy pickles (gibbs:320-343)."""
    import pickle
    mod = RL.load_gibbs_vl()
    key, val = make_proj(7, 768)
    ref = mod.LongTermAttention(**RL.caller_kwargs(64, 0.75, True, key, val))
    orc = O.RectLTM(64, 0.75, *proj_tensors(key, val))
    ks, qs, _ = make_inputs(8, 2, 1, 8 * 32, 768, 32, q_scale=3.0)
    cwd = os.getcwd()
    os.chdir(tmp_path)
    try:
        with torch.no_grad():
            for c in range(2):
                torch.manual_seed(300 + c)
                ref(ks[c], qs[c], new_doc=(c == 0), layer_n=0)
                torch.manual_seed(300 + c)
                u = torch.rand(1, 512, dtype=torch.float64)
                orc.forward(ks[c], qs[c], c == 0, u)
                with open("alphas_uniform", "rb") as f:
                    want = pickle.load(f)
                got = O.rect_density_alphas(orc, orc.tables(8))
                assert got.shape == want.shape == (32, 1, 12, 768)
                assert torch.equal(got, want), f"chunk {c}"
    finally:
        os.chdir(cwd)


@needs_reference
@pytest.mark.parametrize("alpha,N,L", [(0.5, 64, 8), (0.9, 256, 32)])
def test_caller_cross_attention_with_ltm_blend(alpha, N, L, tmp_path):
    """C1 + N1: the oracle's restatement of BertSelfAttention's cross-attention branch (short-term softmax
    attention + (1-alpha) LTM, Qformer.py:197-310) against the real caller module."""
    Q = RL.load_qformer_vl()
    cfg = RL.bert_config(N, 0.75, alpha)
    torch.manual_seed(11)
    att = Q.BertSelfAttention(cfg, is_cross_attention=True).eval()
    orc = O.CrossAttentionLTM(N, 0.75, alpha, att.query.weight.detach(), att.query.bias.detach(),
                              att.key.weight.detach(), att.key.bias.detach(), att.value.weight.detach(),
                              att.value.bias.detach())
    g = torch.Generator().manual_seed(12)
    cwd = os.getcwd()
    os.chdir(tmp_path)
    try:
        with torch.no_grad():
            for c in range(3):
                hidden = torch.randn(1, 32, 768, generator=g)
                enc = torch.randn(1, L * 32, 768, generator=g)
                torch.manual_seed(500 + c)
                want = att(hidden, position_embedding_ext=torch.zeros(1), layer=0, encoder_hidden_states=enc,
                           new_video=(c == 0))[0]
                torch.manual_seed(500 + c)
                u = torch.rand(1, 512, dtype=torch.float64)
                got = orc.forward(hidden, enc, c == 0, u)
                assert torch.equal(got, want), f"chunk {c}: {float((got - want).abs().max())}"
    finally:
        os.chdir(cwd)
