"""fp16 / bfloat16 chunks through every entry point of the batched variant-R engine: the bounded-grid 16-bit pooling
kernel, `step_overlapped` (lock-step and ragged), `prefetch` + `step`, and `step_host` give the bits `step` gives on
the same 16-bit chunk; the engine tracks the oracle run on the up-cast chunks; bad chunks are refused before any
state changes."""
import numpy as np
import pytest
import torch

from oracle import ltm_oracle as O
from tests.helpers import TOL_CTX, compare_draws, make_proj, proj_tensors, relerr

pytestmark = pytest.mark.gpu

DTYPES = [torch.float16, torch.bfloat16]
TIE = 1e-3


@pytest.fixture(scope="module")
def dev(cuda_device):
    return cuda_device


def _engines(dev, N, e=768, T=32, n=2, seed=41, **kw):
    from infinite_video_b200.batched import BatchedRectLTM
    key, val = make_proj(seed, e)
    return [BatchedRectLTM(N, .75, *proj_tensors(key, val), tokens_per_frame=T, device=dev, **kw) for _ in range(n)], \
        (key, val)


def _chunks(dev, C, Bv, L, dtype, T=32, e=768, Q=32, seed=0):
    g = torch.Generator(device=dev).manual_seed(seed)
    ks = [torch.randn(Bv, L * T, e, generator=g, device=dev).to(dtype) for _ in range(C)]
    qs = [torch.randn(Bv, Q, 768, generator=g, device=dev) for _ in range(C)]
    us = [torch.rand(Bv, 512, generator=g, device=dev, dtype=torch.float64) for _ in range(C)]
    return ks, qs, us


def _state(eng, ctx):
    last = eng.last
    kv = last["KV"] if last["KV"] is not None else last["V"]
    return [ctx, eng.B_past, kv, eng._hist, last["idx"], last["b"]]


def _assert_same(a, b, ctx_a, ctx_b, what):
    names = ["ctx", "B_past", "K|V", "hist", "idx", "b"]
    for n, x, y in zip(names, _state(a, ctx_a), _state(b, ctx_b)):
        assert torch.equal(x, y), f"{what}: {n} differs"


def _sentinel(*engs):
    # draws of a first chunk are not written: the same sentinel in both engines keeps the comparison like for like
    for eng in engs:
        eng.last["idx"].fill_(-7)
        eng.last["b"].fill_(-7)


def _lockstep_flags(c, Bv, dev):
    if c == 0:
        return True
    if c == 2:
        return torch.tensor([v % 2 == 0 for v in range(Bv)], device=dev)     # per-video new documents
    return False


# --------------------------------------------------------------------------- kernel
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("Bv,L,T,e,splits", [(3, 8, 32, 768, 1), (1, 16, 196, 1024, 5), (2, 5, 32, 776, 2)])
def test_pool_mean_16_grid_is_bit_identical_for_any_grid(dev, dtype, Bv, L, T, e, splits):
    from infinite_video_b200 import _capi as ca
    from infinite_video_b200 import ops
    g = torch.Generator(device=dev).manual_seed(5)
    k = (torch.randn(Bv, L, T, e, generator=g, device=dev) * 3).to(dtype)
    want = ops.pool_mean(k, splits)
    units = Bv * L * splits
    for max_ctas in (0, 1, 7, 150, units, units + 3):
        out = torch.full_like(want, float("nan"))
        ca.check(ca.lib().ltm_pool_mean_16_grid(ca.ptr(k), int(dtype == torch.bfloat16), ca.ptr(out), Bv, L, T, e,
                                                splits, max_ctas, ca.stream_ptr(dev)), "pool_mean_16_grid")
        assert torch.equal(out, want), max_ctas
    torch.cuda.synchronize()


# --------------------------------------------------------------------------- lock-step overlapped step
@pytest.mark.parametrize("dtype,Bv,L,N,pool_ctas", [
    (torch.float16, 3, 8, 64, 0),
    (torch.bfloat16, 3, 8, 64, 0),
    (torch.float16, 3, 8, 64, 5),
    (torch.bfloat16, 2, 32, 256, 11),
    (torch.float16, 128, 256, 256, 0),                 # the NExT-QA batch of the benchmark
])
def test_overlapped_equals_step(dev, dtype, Bv, L, N, pool_ctas):
    (a, b), _ = _engines(dev, N)
    b.pool_ctas = pool_ctas
    C = 5
    ks, qs, us = _chunks(dev, C, Bv, L, dtype, seed=Bv + L)
    with torch.no_grad():
        for c in range(C):
            nd = _lockstep_flags(c, Bv, dev)
            u = us[c] if c else None
            x = a.step(ks[c], qs[c], u, new_doc=nd)
            y = b.step_overlapped(ks[c], qs[c], u, new_doc=nd, k_next=ks[c + 1] if c + 1 < C else None)
            if c == 0:
                _sentinel(a, b)
            _assert_same(a, b, x, y, f"chunk {c}")
    assert not b._pref
    torch.cuda.synchronize()


def _ragged_schedule(Bv, L, C, seed):
    """Per-chunk lengths (0 = idle) and host new_doc flags: idle slots, a slot emptied and refilled, restarts."""
    rng = np.random.RandomState(seed)
    mem = np.zeros(Bv, bool)
    lens, nds = [], []
    for c in range(C):
        ln = rng.randint(2, L + 1, Bv)
        ln[0] = L
        if c in (1, 2):
            ln[1] = 0                                  # idle for two chunks ...
        nd = np.zeros(Bv, bool) if c else np.ones(Bv, bool)
        if c == 3:
            nd[1] = True                               # ... then refilled with a new video
        if c == 2:
            ln[2] = 0
            nd[2] = True                               # slot cleared
        nd |= (ln > 0) & ~mem
        mem = np.where(nd, ln > 0, mem)
        lens.append(ln.tolist())
        nds.append(nd.tolist())
    return lens, nds


@pytest.mark.parametrize("dtype", DTYPES)
def test_ragged_overlapped_equals_ragged_step(dev, dtype):
    Bv, L, N, C = 4, 16, 64, 5
    (a, b), _ = _engines(dev, N)
    ks, qs, us = _chunks(dev, C, Bv, L, dtype, seed=3)
    lens, nds = _ragged_schedule(Bv, L, C, 11)
    for c in range(C):
        for v, Lv in enumerate(lens[c]):
            ks[c][v, Lv * 32:] = float("nan")          # padding is never read
    with torch.no_grad():
        for c in range(C):
            x = a.step(ks[c], qs[c], us[c], new_doc=nds[c], lengths=lens[c])
            nxt = c + 1 < C
            y = b.step_overlapped(ks[c], qs[c], us[c], new_doc=nds[c], lengths=lens[c],
                                  k_next=ks[c + 1] if nxt else None, next_lengths=lens[c + 1] if nxt else None)
            if c == 0:
                _sentinel(a, b)
            assert not torch.isnan(y).any()
            _assert_same(a, b, x, y, f"chunk {c}")
    torch.cuda.synchronize()


# --------------------------------------------------------------------------- prefetch
@pytest.mark.parametrize("dtype", DTYPES)
def test_prefetch_then_step_matches_and_mixes_with_fp32(dev, dtype):
    """prefetch(k16) + step(k16) == step(k16) and consumes the prefetch; a pending 16-bit prefetch is not taken by an
    fp32 chunk and vice versa.  bin_pool=True: fp32 update chunks are pooled per bin, 16-bit ones never are."""
    Bv, L, N = 2, 256, 256
    (a, b), _ = _engines(dev, N, bin_pool=True)
    order = [dtype, torch.float32, dtype, dtype, torch.float32]
    ks, qs, us = _chunks(dev, 5, Bv, L, torch.float32, seed=8)
    ks = [k.to(dt) for k, dt in zip(ks, order)]
    out = {}

    def step_b(c):
        out[c] = b.step(ks[c], qs[c], us[c] if c else None, new_doc=(c == 0))
        if c == 0:
            _sentinel(b)

    with torch.no_grad():
        x = a.step(ks[0], qs[0], new_doc=True)
        _sentinel(a)
        b.prefetch(ks[0], 32)
        step_b(0)
        assert not b._pref
        _assert_same(a, b, x, out[0], "chunk 0")
        b.prefetch(ks[2], 32, update=True)            # 16-bit prefetch, then an fp32 chunk
        step_b(1)
        assert len(b._pref) == 1
        x = a.step(ks[1], qs[1], us[1])
        _assert_same(a, b, x, out[1], "chunk 1")
        step_b(2)
        assert not b._pref
        x = a.step(ks[2], qs[2], us[2])
        _assert_same(a, b, x, out[2], "chunk 2")
        b.prefetch(ks[4], 32, update=True)            # fp32 prefetch (per bin), then a 16-bit chunk
        step_b(3)
        assert len(b._pref) == 1 and b._pref[0]["binned"]
        x = a.step(ks[3], qs[3], us[3])
        _assert_same(a, b, x, out[3], "chunk 3")
        step_b(4)
        assert not b._pref
        x = a.step(ks[4], qs[4], us[4])
        _assert_same(a, b, x, out[4], "chunk 4")
    torch.cuda.synchronize()


# --------------------------------------------------------------------------- host buffers
def test_step_host_with_16_bit_chunks(dev):
    """Pinned fp16 / bf16 / fp32 host chunks, the storage changing between calls: step_host == step on the device
    copies, bit for bit."""
    Bv, L, N = 3, 8, 64
    (a, b), _ = _engines(dev, N)
    order = [torch.float16, torch.float16, torch.bfloat16, torch.float32, torch.float16]
    ks, qs, us = _chunks(dev, len(order), Bv, L, torch.float32, seed=12)
    ks = [k.to(dt) for k, dt in zip(ks, order)]
    with torch.no_grad():
        for c in range(len(order)):
            u = us[c] if c else None
            x = a.step(ks[c], qs[c], u, new_doc=(c == 0))
            y = b.step_host(ks[c].cpu().pin_memory(), qs[c].cpu().pin_memory(),
                            u.cpu().pin_memory() if u is not None else None, new_doc=(c == 0))
            torch.cuda.synchronize()
            if c == 0:
                _sentinel(a, b)
            _assert_same(a, b, x, y.to(dev), f"chunk {c} ({order[c]})")
            assert b._workspace(Bv, L, 32)["k_dev"].dtype == order[c]


# --------------------------------------------------------------------------- oracle
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("name,N,L,Bv,C,T,e,Q", [
    ("nextqa", 256, 256, 4, 4, 32, 768, 32),
    ("videochat2", 64, 16, 2, 3, 196, 1024, 96),
])
def test_overlapped_16_bit_tracks_oracle_on_upcast_chunks(dev, dtype, name, N, L, Bv, C, T, e, Q):
    (eng,), (key, val) = _engines(dev, N, e=e, T=T, n=1, seed=77)
    orcs = [O.RectLTM(N, .75, *proj_tensors(key, val), tokens_per_frame=T, rebuild_tables=False) for _ in range(Bv)]
    ks, qs, us = _chunks(dev, C, Bv, L, dtype, T=T, e=e, Q=Q, seed=78)
    worst = dict(B=0.0, ctx=0.0, flips=0, draws=0)
    with torch.no_grad():
        for c in range(C):
            u = us[c] if c else None
            got = eng.step_overlapped(ks[c], qs[c], u, new_doc=(c == 0), k_next=ks[c + 1] if c + 1 < C else None)
            k32, q32 = ks[c].float().cpu(), qs[c].cpu()
            b_got = eng.last["b"].cpu().long() if c else None
            want = torch.cat([orcs[v].forward(k32[v:v + 1], q32[v:v + 1], c == 0, u[v:v + 1].cpu() if c else None,
                                              b_override=b_got[v:v + 1] if c else None) for v in range(Bv)])
            if c:
                f, d = compare_draws(b_got, torch.cat([o.last["b_own"] for o in orcs]), u.cpu(),
                                     torch.cat([o.last["p"] for o in orcs]), TIE)
                worst["flips"] += f
                worst["draws"] += d
            worst["B"] = max(worst["B"], relerr(eng.B_past, torch.cat([o.B_past for o in orcs])))
            worst["ctx"] = max(worst["ctx"], relerr(got, want))
    print(f"[flips] half_{name}_{str(dtype)[6:]}: {worst['flips']} of {worst['draws']} draws, "
          f"B {worst['B']:.2e}, ctx {worst['ctx']:.2e}")
    assert worst["B"] <= 1e-5 and worst["ctx"] <= TOL_CTX, worst


# --------------------------------------------------------------------------- refusals
def _snapshot(eng):
    return (eng.has_state, eng._cur, eng.Bv, len(eng._pref), eng.B_past.clone() if eng.B_past is not None else None)


def _same_snapshot(s, t):
    assert s[:4] == t[:4]
    assert (s[4] is None) == (t[4] is None) and (s[4] is None or torch.equal(s[4], t[4]))


@pytest.mark.parametrize("e", [768, 772])
def test_bad_chunks_are_refused_before_any_state_change(dev, e):
    """float64 chunks, 16-bit chunks of a width that is not a multiple of 8 and queries that are not float32 raise a
    ValueError from every entry point before the engine changes (width 768: after a first chunk, which the engine
    then continues as if nothing had been asked)."""
    Bv, L = 2, 8
    (eng,), _ = _engines(dev, 64, e=e, n=1)
    ks, qs, us = _chunks(dev, 2, Bv, L, torch.float32, e=e, seed=21)
    if e % 8 == 0:
        eng.step(ks[0], qs[0], new_doc=True)
        torch.cuda.synchronize()
    bad = [ks[1].double()] + ([ks[1].half(), ks[1].bfloat16()] if e % 8 else [])
    good16 = [] if e % 8 else [ks[1].half()]
    snap = _snapshot(eng)
    for k in bad:
        with pytest.raises(ValueError):
            eng.step(k, qs[1], us[1])
        with pytest.raises(ValueError):
            eng.step_overlapped(k, qs[1], us[1])
        with pytest.raises(ValueError):
            eng.step_overlapped(ks[1], qs[1], us[1], k_next=k)
        with pytest.raises(ValueError):
            eng.prefetch(k, 32)
        with pytest.raises(ValueError):
            eng.step_host(k.cpu(), qs[1].cpu(), us[1].cpu())
        _same_snapshot(snap, _snapshot(eng))
    for q in (qs[1].half(), qs[1].double()):                   # queries stay float32
        for k in [ks[1]] + good16:
            with pytest.raises(ValueError):
                eng.step(k, q, us[1])
            with pytest.raises(ValueError):
                eng.step_overlapped(k, q, us[1])
            with pytest.raises(ValueError):
                eng.step_host(k.cpu(), q.cpu(), us[1].cpu())
            _same_snapshot(snap, _snapshot(eng))
    if e % 8 == 0:
        (ref,), _ = _engines(dev, 64, e=e, n=1)
        ref.step(ks[0], qs[0], new_doc=True)
        want = ref.step(ks[1], qs[1], us[1])
        got = eng.step(ks[1], qs[1], us[1])
        assert torch.equal(got, want) and torch.equal(eng.B_past, ref.B_past)
    torch.cuda.synchronize()
