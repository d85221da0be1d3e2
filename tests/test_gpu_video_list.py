"""Chunks given per video (`BatchedRectLTM.step(k=[...], chunk_frames=L)`): every frame pooled where it lives, through
a per-video pointer table.  Against the padded ragged step (bit for bit, through every entry point), against one
oracle per video (`split_videos` + `consolidate_video`), and the validation of the entries."""
import gc

import numpy as np
import pytest
import torch

from oracle import ltm_oracle as O
from tests.helpers import TOL_CTX, compare_draws, make_proj, proj_tensors, relerr

pytestmark = pytest.mark.gpu

E, QN, S, T = 768, 32, 512, 32
DTYPES = (torch.float32, torch.float16, torch.bfloat16)
FORMS = ("separate", "video", "packed")
NAN = float("nan")


@pytest.fixture(scope="module")
def dev(cuda_device):
    return cuda_device


def _engine(dev, N, seed=31, **kw):
    from infinite_video_b200.batched import BatchedRectLTM
    key, val = make_proj(seed, E)
    return BatchedRectLTM(N, .75, *proj_tensors(key, val), tokens_per_frame=T, device=dev, **kw), (key, val)


def _entries(parts, dt, dev, form):
    """Per-video chunk parts (CPU [n_v*T, e] or None) as list entries on the device, in one of three layouts; the
    memory next to every entry holds NaN (padding that must never be read)."""
    if form == "separate":
        return [None if p is None else p.to(dev, dt) for p in parts]
    if form == "video":                         # each chunk a view into a longer per-video tensor
        out = []
        for p in parts:
            if p is None:
                out.append(None)
                continue
            big = torch.full((p.shape[0] + 2 * T, E), NAN, device=dev, dtype=dt)
            big[T:T + p.shape[0]] = p.to(dev, dt)
            out.append(big[T:T + p.shape[0]])
        return out
    rows = sum(p.shape[0] + T for p in parts if p is not None) + T      # one packed tensor, NaN rows in between
    buf = torch.full((rows, E), NAN, device=dev, dtype=dt)
    out, r = [], T
    for p in parts:
        if p is None:
            out.append(None)
            continue
        buf[r:r + p.shape[0]] = p.to(dev, dt)
        out.append(buf[r:r + p.shape[0]])
        r += p.shape[0] + T
    return out


def _padded(parts, L, dt, dev):
    k = torch.zeros(len(parts), L * T, E, dtype=dt)
    for v, p in enumerate(parts):
        if p is not None:
            k[v, :p.shape[0]] = p.to(dt)
    return k.to(dev)


def _plan(L):
    """Per-chunk lengths and host new_doc flags over five chunks of four slots: idle slots, and slot 1 refilled."""
    lens = [[L, 5, 2, L], [3, 0, L, 2], [L, 4, 0, 6], [2, L, 7, 0], [0, 3, L, L]]
    nd = [[True] * 4, [False] * 4, [False, True, False, False], [False] * 4, [False] * 4]
    return lens, nd


def _chunks(seed, L, n=5):
    g = torch.Generator().manual_seed(seed)
    lens, nd = _plan(L)
    parts = [[torch.randn(Lv * T, E, generator=g) if Lv else None for Lv in lens[c]] for c in range(n)]
    qs = [torch.randn(4, QN, 768, generator=g) for _ in range(n)]
    us = [torch.rand(4, S, dtype=torch.float64, generator=g) for _ in range(n)]
    return lens, nd, parts, qs, us


def _same(a, b, ya, yb, c, drew=()):
    """Bits of two engines after the same step; `drew`: the slots whose re-sampling ran (the draw buffers of the
    others hold whatever an earlier step left there)."""
    assert torch.isfinite(yb).all(), c
    assert torch.equal(ya, yb), c
    assert torch.equal(a.B_past, b.B_past), c
    for n in ("KV", "V"):
        if a.last.get(n) is not None:
            assert torch.equal(a.last[n], b.last[n]), (c, n)
    for n in ("b", "ts", "idx"):
        for v in drew:
            assert torch.equal(a.last[n][v], b.last[n][v]), (c, n, v)


# --------------------------------------------------------------------------- list step == padded ragged step
@pytest.mark.parametrize("dt", DTYPES, ids=["fp32", "fp16", "bf16"])
@pytest.mark.parametrize("N,L,kw", [
    (64, 8, {}),
    (256, 16, dict(tc_attn=False)),
    (512, 16, {}),
    (64, 8, dict(kv_dtype="fp32")),
])
def test_list_step_equals_padded_ragged_step(dev, dt, N, L, kw):
    a, _ = _engine(dev, N, keep_scores=True, **kw)
    b, _ = _engine(dev, N, keep_scores=True, **kw)
    lens, nd, parts, qs, us = _chunks(5, L)
    with torch.no_grad():
        for c in range(len(lens)):
            q, u = qs[c].to(dev), us[c].to(dev) if c else None
            ya = a.step(_padded(parts[c], L, dt, dev), q, u, new_doc=nd[c], lengths=lens[c])
            yb = b.step(_entries(parts[c], dt, dev, FORMS[c % 3]), q, u, new_doc=nd[c], chunk_frames=L)
            _same(a, b, ya, yb, c, [v for v in range(4) if c and lens[c][v] and not nd[c][v]])
            for v, Lv in enumerate(lens[c]):
                if Lv == 0:
                    assert not yb[v].any()
        assert torch.equal(a.density(), b.density())
        with pytest.raises(RuntimeError):
            b.x_past()


# --------------------------------------------------------------------------- every entry point, prefetches consumed
@pytest.mark.parametrize("dt", DTYPES, ids=["fp32", "fp16", "bf16"])
def test_every_entry_point_same_bits(dev, dt):
    N, L = 64, 8
    lens, nd, parts, qs, us = _chunks(7, L)
    C = len(lens)
    ref, _ = _engine(dev, N)
    with torch.no_grad():
        want = []
        for c in range(C):
            want.append(ref.step(_padded(parts[c], L, dt, dev), qs[c].to(dev), us[c].to(dev) if c else None,
                                 new_doc=nd[c], lengths=lens[c]))
        B_want = ref.B_past.clone()

        # step_overlapped: list -> padded -> list -> list -> list, each k the k_next of the call before
        b, _ = _engine(dev, N)
        calls = []
        pf = b.prefetch
        b.prefetch = lambda *x, **kw: (calls.append(1), pf(*x, **kw))[1]
        ks = [_entries(parts[c], dt, dev, FORMS[c % 3]) if c != 1 else _padded(parts[c], L, dt, dev)
              for c in range(C)]
        for c in range(C):
            nxt = ks[c + 1] if c + 1 < C else None
            y = b.step_overlapped(ks[c], qs[c].to(dev), us[c].to(dev) if c else None, new_doc=nd[c], k_next=nxt,
                                  lengths=lens[c] if c == 1 else None,
                                  next_lengths=lens[c + 1] if c + 1 == 1 else None, chunk_frames=L)
            assert torch.equal(y, want[c]), c
            assert len(b._pref) == (1 if nxt is not None else 0), c
        assert len(calls) == 1                      # only the first chunk was pooled on arrival
        assert torch.equal(b.B_past, B_want)

        # prefetch + step
        p, _ = _engine(dev, N)
        for c in range(C):
            k = _entries(parts[c], dt, dev, FORMS[(c + 1) % 3])
            p.prefetch(k, QN, chunk_frames=L)
            y = p.step(k, qs[c].to(dev), us[c].to(dev) if c else None, new_doc=nd[c], chunk_frames=L)
            assert not p._pref, c                   # consumed, not pooled again
            assert torch.equal(y, want[c]), c
        assert torch.equal(p.B_past, B_want)

        # pool + step(pooled=): the packed frames of the list
        s, _ = _engine(dev, N)
        for c in range(C):
            k = _entries(parts[c], dt, dev, FORMS[(c + 2) % 3])
            x = s.pool(k, chunk_frames=L)
            assert x.shape[0] == sum(lens[c])
            xr = ref.pool(_padded(parts[c], L, dt, dev), lengths=lens[c])
            assert torch.equal(x, xr), c
            y = s.step(k, qs[c].to(dev), us[c].to(dev) if c else None, new_doc=nd[c], pooled=x, chunk_frames=L)
            assert torch.equal(y, want[c]), c
        assert torch.equal(s.B_past, B_want)


# --------------------------------------------------------------------------- the side stream's reads are protected
def test_dropped_entries_are_not_reused_before_pooled(dev):
    N, L, Bv = 64, 64, 16
    g = torch.Generator().manual_seed(11)
    lens0 = [L] * Bv
    lens1 = [L - (v % 5) for v in range(Bv)]
    c0 = [torch.randn(n * T, E, generator=g) for n in lens0]
    c1 = [torch.randn(n * T, E, generator=g) for n in lens1]
    q0, q1 = (torch.randn(Bv, QN, 768, generator=g).to(dev) for _ in range(2))
    u1 = torch.rand(Bv, S, dtype=torch.float64, generator=g).to(dev)
    ref, _ = _engine(dev, N)
    b, _ = _engine(dev, N)
    with torch.no_grad():
        ref.step(_padded(c0, L, torch.float32, dev), q0, new_doc=True, lengths=lens0)
        want = ref.step(_padded(c1, L, torch.float32, dev), q1, u1, lengths=lens1)
        nxt = [p.to(dev) for p in c1]
        b.step_overlapped([p.to(dev) for p in c0], q0, new_doc=True, k_next=nxt, chunk_frames=L)
        ent = b._pref[-1]
        del nxt                                      # the caller drops the tensors it handed over ...
        gc.collect()
        junk = [torch.full((n * T, E), NAN, device=dev) for n in lens1]     # ... and refills memory on its stream
        torch.cuda.synchronize()
        ws = next(iter(b._ws.values()))
        frames = sum(lens1)
        splits = b._splits(frames)
        got = ws["xbufs"][ent["buf"]][:frames * splits * E].view(frames, splits, E)
        again = [p.to(dev) for p in c1]
        assert torch.equal(got, b.pool(again, chunk_frames=L))               # the pooling read the chunk, not junk
        y = b.step_overlapped(again, q1, u1, chunk_frames=L)
        assert torch.equal(y, want)
        del junk


# --------------------------------------------------------------------------- whole videos against the oracle
def _videos(seed, frames):
    g = torch.Generator().manual_seed(seed)
    return [torch.randn(F * T, E, generator=g) for F in frames]


def test_split_videos_consolidate_matches_oracle(dev):
    from infinite_video_b200.video import consolidate_video, split_videos
    N, L, frames = 64, 8, (20, 7, 13, 2, 16)
    Bv = len(frames)
    vids = _videos(13, frames)
    chunks = split_videos([v.to(dev) for v in vids], L, T)
    C = len(chunks)
    g = torch.Generator().manual_seed(17)
    qs = [torch.randn(Bv, QN, 768, generator=g) for _ in range(C)]
    us = [torch.rand(Bv, S, dtype=torch.float64, generator=g) for _ in range(C)]
    eng, kv = _engine(dev, N)
    orcs = [O.RectLTM(N, .75, *proj_tensors(*kv), tokens_per_frame=T, rebuild_tables=False) for _ in range(Bv)]
    worst = dict(B=0.0, ctx=0.0, flips=0, draws=0)
    wants = {}

    def check(c):                                   # the state the engine left after chunk c, video by video
        for v in range(Bv):
            if chunks[c][v] is None:
                continue
            n = chunks[c][v].shape[0]
            upd = c > 0
            b_got = eng.last["b"][v:v + 1].cpu().long() if upd else None
            wants[c, v] = orcs[v].forward(vids[v][c * L * T:c * L * T + n].unsqueeze(0), qs[c][v:v + 1], not upd,
                                          us[c][v:v + 1] if upd else None, b_override=b_got)
            if upd:
                f, d = compare_draws(b_got, orcs[v].last["b_own"], us[c][v:v + 1], orcs[v].last["p"], 1e-3)
                worst["flips"] += f
                worst["draws"] += d
            worst["B"] = max(worst["B"], relerr(eng.B_past[v:v + 1], orcs[v].B_past))

    def queries(li, c, prev):
        if c:
            check(c - 1)
        return qs[c].to(dev)

    with torch.no_grad():
        out = consolidate_video([eng], chunks, queries, [[u.to(dev) for u in us]], chunk_frames=L)[0]
        check(C - 1)
    for (c, v), want in wants.items():
        worst["ctx"] = max(worst["ctx"], relerr(out[c][v:v + 1], want))
    for c in range(C):
        for v in range(Bv):
            if chunks[c][v] is None:
                assert not out[c][v].any()
    assert worst["B"] < 1e-5 and worst["ctx"] < TOL_CTX, worst
    assert worst["flips"] <= 0.01 * max(worst["draws"], 1), worst


def test_consolidate_video_list_equals_padded(dev):
    from infinite_video_b200.video import consolidate_video, split_videos
    N, L, frames = 64, 8, (20, 7, 13, 2)
    Bv = len(frames)
    vids = _videos(19, frames)
    chunks = split_videos([v.to(dev) for v in vids], L, T)
    C = len(chunks)
    lengths = [[0 if x is None else x.shape[0] // T for x in ch] for ch in chunks]
    padded = [_padded([None if x is None else x.cpu() for x in ch], L, torch.float32, dev) for ch in chunks]
    g = torch.Generator().manual_seed(23)
    qs = [[torch.randn(Bv, QN, 768, generator=g).to(dev) for _ in range(C)] for _ in range(2)]
    us = [[torch.rand(Bv, S, dtype=torch.float64, generator=g).to(dev) for _ in range(C)] for _ in range(2)]
    with torch.no_grad():
        for reduce in (None, "mean"):
            a = [_engine(dev, N, seed=s)[0] for s in (1, 2)]
            b = [_engine(dev, N, seed=s)[0] for s in (1, 2)]
            ya = consolidate_video(a, padded, qs, us, reduce=reduce, lengths=lengths)
            yb = consolidate_video(b, chunks, qs, us, reduce=reduce, chunk_frames=L)
            for la, lb in zip(ya, yb):
                if reduce is None:
                    assert all(torch.equal(x, y) for x, y in zip(la, lb))
                else:
                    assert torch.equal(la, lb)


# --------------------------------------------------------------------------- validation leaves the engine untouched
def test_bad_entries_raise_and_leave_engine_untouched(dev):
    N, L = 64, 8
    lens, nd, parts, qs, us = _chunks(29, L, n=2)
    a, _ = _engine(dev, N)
    b, _ = _engine(dev, N)
    with torch.no_grad():
        k0 = _entries(parts[0], torch.float32, dev, "packed")
        ya = a.step(k0, qs[0].to(dev), new_doc=True, chunk_frames=L)
        yb = b.step(k0, qs[0].to(dev), new_doc=True, chunk_frames=L)
        assert torch.equal(ya, yb)
        good = _entries(parts[1], torch.float32, dev, "separate")       # lengths [3, 0, 8, 2]
        q, u = qs[1].to(dev), us[1].to(dev)
        flat = torch.zeros(8 * T * E + 4, device=dev)

        def with_entry(v, t):
            k = list(good)
            k[v] = t
            return k

        bad = {
            "device": with_entry(0, good[0].cpu()),
            "dtype": with_entry(2, good[2].half()),
            "float64": with_entry(0, good[0].double()),
            "width": with_entry(0, torch.zeros(3 * T, E - 8, device=dev)),
            "tokens": with_entry(0, torch.zeros(3 * T + 1, E, device=dev)),
            "one frame": with_entry(3, torch.zeros(T, E, device=dev)),
            "too long": with_entry(3, torch.zeros((L + 1) * T, E, device=dev)),
            "strides": with_entry(0, torch.zeros(3 * T, 2 * E, device=dev)[:, :E]),
            "aligned": with_entry(0, flat[1:1 + 3 * T * E].view(3 * T, E)),
            "not a tensor": with_entry(0, 3.0),
        }
        for name, k in bad.items():
            with pytest.raises(ValueError):
                a.step(k, q, u, chunk_frames=L)
            with pytest.raises(ValueError):
                a.step_overlapped(k, q, u, chunk_frames=L)
            with pytest.raises(ValueError):
                a.step_overlapped(_entries(parts[1], torch.float32, dev, "separate"), q, u, k_next=k,
                                  chunk_frames=L)
            with pytest.raises(ValueError):
                a.prefetch(k, QN, chunk_frames=L)
            with pytest.raises(ValueError):
                a.pool(k, chunk_frames=L)
        with pytest.raises(ValueError, match="lengths"):
            a.step(good, q, u, lengths=lens[1], chunk_frames=L)
        with pytest.raises(ValueError, match="chunk_frames"):
            a.step(good, q, u)
        with pytest.raises(ValueError, match="chunk_frames"):
            a.step(_padded(parts[1], L, torch.float32, dev), q, u, lengths=lens[1], chunk_frames=L)
        with pytest.raises(ValueError, match="with_half"):
            a.pool(good, with_half=True, chunk_frames=L)
        with pytest.raises(ValueError):
            a.step_overlapped(good, q, u, k_next=good[:3], chunk_frames=L)              # other batch size
        assert not a._pref
        ya = a.step(good, q, u, chunk_frames=L)
        yb = b.step(good, q, u, chunk_frames=L)
        assert torch.equal(ya, yb) and torch.equal(a.B_past, b.B_past)
        assert torch.equal(a.last["KV"], b.last["KV"])
        assert np.array_equal(a._slots, b._slots)
