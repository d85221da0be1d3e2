"""Ragged batches of variant R: per-video chunk lengths and idle slots in one batched step
(`BatchedRectLTM.step(..., lengths=...)`), against the lock-step step and against one oracle per video."""
import numpy as np
import pytest
import torch

from oracle import ltm_oracle as O
from tests.helpers import TOL_CTX, compare_draws, make_proj, proj_tensors, relerr

pytestmark = pytest.mark.gpu

TIE = {"tf32": 1e-3, "tf32x3": 2e-5}
E, QN, S = 768, 32, 512


@pytest.fixture(scope="module")
def dev(cuda_device):
    return cuda_device


def _engine(dev, N, tau=.75, T=32, seed=31, **kw):
    from infinite_video_b200.batched import BatchedRectLTM
    key, val = make_proj(seed, E)
    kw.setdefault("keep_scores", True)
    return BatchedRectLTM(N, tau, *proj_tensors(key, val), tokens_per_frame=T, device=dev, **kw), (key, val)


def _oracle(N, tau, kv, T=32, spacing="linear", precision="tf32"):
    return O.RectLTM(N, tau, *proj_tensors(*kv), tokens_per_frame=T, rebuild_tables=False, spacing=spacing)


class _Track:
    """One oracle per video id; each sees only its own frames and never an idle step."""

    def __init__(self, N, tau, kv, T=32, spacing="linear", tie=TIE["tf32"]):
        self.args, self.orcs, self.tie = (N, tau, kv, T, spacing), {}, tie
        self.T = T
        self.worst = dict(B=0.0, ctx=0.0, flips=0, draws=0)

    def check(self, eng, vid, slot, k, q, u, Lv, first, ctx):
        if first:
            self.orcs[vid] = _oracle(*self.args)
        orc = self.orcs[vid]
        upd = not first and eng.sticky
        b_got = eng.last["b"][slot:slot + 1].cpu().long() if upd else None
        want = orc.forward(k[slot:slot + 1, :Lv * self.T].cpu(), q[slot:slot + 1].cpu(), first,
                           u[slot:slot + 1].cpu() if upd else None, b_override=b_got)
        if upd:
            f, d = compare_draws(b_got, orc.last["b_own"], u[slot:slot + 1].cpu(), orc.last["p"], self.tie)
            self.worst["flips"] += f
            self.worst["draws"] += d
        self.worst["B"] = max(self.worst["B"], relerr(eng.B_past[slot:slot + 1], orc.B_past))
        self.worst["ctx"] = max(self.worst["ctx"], relerr(ctx[slot:slot + 1], want))

    def assert_ok(self):
        w = self.worst
        assert w["B"] < 1e-5 and w["ctx"] < TOL_CTX, w
        assert w["flips"] <= 0.01 * max(w["draws"], 1), w


def _chunk(g, Bv, L, T=32, lens=None, fill=0.0):
    k = torch.randn(Bv, L * T, E, generator=g)
    if lens is not None:
        for v, Lv in enumerate(lens):
            k[v, Lv * T:] = fill
    return k, torch.randn(Bv, QN, 768, generator=g), torch.rand(Bv, S, dtype=torch.float64, generator=g)


# --------------------------------------------------------------------------- equal lengths == lock-step, bit for bit
@pytest.mark.parametrize("N,L,kw", [
    (64, 8, {}),
    (256, 32, {}),
    (512, 16, {}),
    (64, 8, dict(kv_dtype="fp32")),
    (64, 8, dict(precision="tf32x3")),
    (256, 16, dict(tc_attn=False)),                     # transposed-key attention
    (64, 8, dict(fast_attn=False)),                     # generic attention
])
def test_equal_lengths_equal_lockstep(dev, N, L, kw):
    Bv, C = 3, 3
    a, _ = _engine(dev, N, bin_pool=False, **kw)
    b, _ = _engine(dev, N, bin_pool=False, **kw)
    g = torch.Generator().manual_seed(5)
    with torch.no_grad():
        for c in range(C):
            k, q, u = (t.to(dev) for t in _chunk(g, Bv, L))
            ya = a.step(k, q, u if c else None, new_doc=(c == 0))
            yb = b.step(k, q, u if c else None, new_doc=(c == 0), lengths=[L] * Bv)
            assert torch.equal(ya, yb), c
            assert torch.equal(a.B_past, b.B_past), c
            if c:
                for n in ("b", "ts", "idx"):
                    assert torch.equal(a.last[n], b.last[n]), (c, n)
            for n in ("KV", "V"):
                if a.last.get(n) is not None:
                    assert torch.equal(a.last[n], b.last[n]), (c, n)


# --------------------------------------------------------------------------- mixed lengths against the oracle
@pytest.mark.parametrize("N,tau,spacing,Lmax", [(100, .5, "linear", 9), (64, .75, "log", 16)])
def test_mixed_lengths_match_oracle(dev, N, tau, spacing, Lmax):
    Bv, C = 4, 4
    eng, kv = _engine(dev, N, tau, spacing=spacing)
    tr = _Track(N, tau, kv, spacing=spacing)
    g = torch.Generator().manual_seed(7)
    rs = np.random.RandomState(3)
    choices = [2, 3, 5, 7, Lmax]
    with torch.no_grad():
        for c in range(C):
            lens = [int(rs.choice(choices)) for _ in range(Bv)]
            lens[c % Bv] = 2 if c % 2 else Lmax
            k, q, u = _chunk(g, Bv, Lmax, lens=lens, fill=float("nan"))
            ctx = eng.step(k.to(dev), q.to(dev), u.to(dev) if c else None, new_doc=(c == 0), lengths=lens)
            assert torch.isfinite(ctx).all()
            for v in range(Bv):
                tr.check(eng, v, v, k, q, u, lens[v], c == 0, ctx)
    tr.assert_ok()


# --------------------------------------------------------------------------- padding is never read
def test_padding_never_read(dev):
    from infinite_video_b200 import ops
    Bv, Lmax, C = 3, 12, 3
    a, _ = _engine(dev, 64)
    b, _ = _engine(dev, 64)
    g = torch.Generator().manual_seed(9)
    with torch.no_grad():
        for c in range(C):
            lens = [[12, 5, 2], [3, 12, 7], [2, 9, 12]][c]
            k, q, u = _chunk(g, Bv, Lmax, lens=lens, fill=0.0)
            kn = k.clone()
            for v, Lv in enumerate(lens):
                kn[v, Lv * 32:] = float("nan")
            ya = a.step(k.to(dev), q.to(dev), u.to(dev) if c else None, new_doc=(c == 0), lengths=lens)
            yb = b.step(kn.to(dev), q.to(dev), u.to(dev) if c else None, new_doc=(c == 0), lengths=lens)
            assert torch.isfinite(yb).all() and torch.equal(ya, yb)
            assert torch.equal(a.B_past, b.B_past)
            # ragged pool rows == lock-step pooling of the same frames with the same splits (fp32 and 16-bit)
            for dt in (torch.float32, torch.float16, torch.bfloat16):
                kd = kn.to(dev, dt)
                x = a.pool(kd, lengths=lens)
                splits, off = x.shape[1], 0
                for v, Lv in enumerate(lens):
                    want = ops.pool_mean(kd[v:v + 1, :Lv * 32].reshape(1, Lv, 32, E), splits)[0]
                    assert torch.equal(x[off:off + Lv], want), (dt, v)
                    off += Lv


# --------------------------------------------------------------------------- idle slots
@pytest.mark.parametrize("kw", [{}, dict(kv_dtype="fp32")])
def test_idle_slots_keep_state(dev, kw):
    Bv, Lmax = 3, 8
    plan = [[8, 8, 8], [8, 0, 5], [0, 6, 8], [7, 7, 0], [8, 0, 0], [2, 4, 3]]
    eng, kv = _engine(dev, 64, **kw)
    tr = _Track(64, .75, kv)
    g = torch.Generator().manual_seed(11)
    with torch.no_grad():
        for c, lens in enumerate(plan):
            k, q, u = _chunk(g, Bv, Lmax, lens=lens, fill=float("nan"))
            for v, Lv in enumerate(lens):
                if Lv == 0:
                    u[v] = float("nan")                  # an idle video's uniforms are never read
            before = None
            if c:
                before = (eng.B_past.clone(), eng.last["KV"].clone(), eng._hist.clone())
            ctx = eng.step(k.to(dev), q.to(dev), u.to(dev) if c else None, new_doc=(c == 0), lengths=lens)
            assert torch.isfinite(ctx).all()
            for v, Lv in enumerate(lens):
                if Lv == 0:
                    assert not ctx[v].any()
                    assert torch.equal(eng.B_past[v], before[0][v])
                    assert torch.equal(eng.last["KV"][v], before[1][v])
                    assert torch.equal(eng._hist[v], before[2][v])
                else:
                    tr.check(eng, v, v, k, q, u, Lv, c == 0, ctx)
    tr.assert_ok()


def test_idle_slot_without_memory_is_defined(dev):
    # a slot that never held memory has zero coefficients and K|V = the bias, whatever the buffers a step writes held
    Bv, Lmax = 3, 8
    eng, _ = _engine(dev, 64)
    g = torch.Generator().manual_seed(13)
    nan = float("nan")
    with torch.no_grad():
        k, q, _u = (t.to(dev) for t in _chunk(g, Bv, Lmax))
        eng.step(k, q, new_doc=True, lengths=[8, 8, 8])           # allocates the buffers
        eng.reset()
        for c, lens in enumerate([[8, 0, 5], [6, 0, 8]]):
            k, q, u = _chunk(g, Bv, Lmax, lens=lens, fill=nan)
            ws = next(iter(eng._ws.values()))
            ws["KVs"][1 - eng._cur].fill_(nan)                    # the buffers this step writes
            ws["B_half"].fill_(nan)
            eng._B[1 - eng._cur].fill_(nan)
            ctx = eng.step(k.to(dev), q.to(dev), u.to(dev) if c else None, new_doc=(c == 0), lengths=lens)
            assert torch.isfinite(ctx).all() and not ctx[1].any()
            assert not eng._B[eng._cur][1].any(), c
            kv = eng.last["KV"][1]
            assert torch.equal(kv, eng.bkv.to(kv.dtype).expand_as(kv)), c


# --------------------------------------------------------------------------- continuous batching through a few slots
def test_continuous_batching(dev):
    slots, Lmax, N = 5, 8, 64
    rs = np.random.RandomState(17)
    videos = []                                           # per video: list of chunk lengths
    for _ in range(13):
        n = int(rs.randint(1, 5))
        videos.append([Lmax] * (n - 1) + [int(rs.choice([2, 3, 5, 7, 8]))])
    eng, kv = _engine(dev, N)
    tr = _Track(N, .75, kv)
    g = torch.Generator().manual_seed(19)
    queue = list(range(len(videos)))
    cur = [None] * slots                                  # (video id, next chunk index)
    done, steps = 0, 0
    with torch.no_grad():
        while done < len(videos):
            lens, nd, who = [0] * slots, [False] * slots, [None] * slots
            for s in range(slots):
                if cur[s] is not None and cur[s][1] >= len(videos[cur[s][0]]):
                    cur[s] = None
                    done += 1
                if cur[s] is None and queue:
                    cur[s] = (queue.pop(0), 0)
                    nd[s] = True                          # refill: new_doc for this slot only
                if cur[s] is not None:
                    vid, ci = cur[s]
                    lens[s], who[s] = videos[vid][ci], (vid, ci)
                    cur[s] = (vid, ci + 1)
            if not any(lens):
                continue
            k, q, u = _chunk(g, slots, Lmax, lens=lens, fill=float("nan"))
            ctx = eng.step(k.to(dev), q.to(dev), u.to(dev), new_doc=nd, lengths=lens)
            steps += 1
            for s in range(slots):
                if who[s] is None:
                    assert not ctx[s].any()
                else:
                    tr.check(eng, who[s][0], s, k, q, u, lens[s], who[s][1] == 0, ctx)
    assert steps >= 6 and set(tr.orcs) == set(range(len(videos)))
    tr.assert_ok()


# --------------------------------------------------------------------------- production shape, overlapped == plain
def test_production_shape_overlapped_equals_step(dev):
    Bv, Lmax, N, C = 128, 256, 256, 3
    rs = np.random.RandomState(23)
    plan = []
    for c in range(C):
        lens = rs.randint(2, Lmax + 1, size=Bv)
        lens[rs.rand(Bv) < 0.1] = 0
        lens[0], lens[1] = Lmax, 2
        plan.append([int(x) for x in lens])
    g = torch.Generator(device=dev).manual_seed(29)
    ks = [torch.randn(Bv, Lmax * 32, E, device=dev, generator=g) for _ in range(C)]
    qs = [torch.randn(Bv, QN, 768, device=dev, generator=g) for _ in range(C)]
    us = [torch.rand(Bv, S, dtype=torch.float64, device=dev, generator=g) for _ in range(C)]
    a, kv = _engine(dev, N, keep_scores=False)
    b, _ = _engine(dev, N, keep_scores=False)
    sample = [0, 1] + [int(x) for x in rs.choice(np.arange(2, Bv), 6, replace=False)]
    tr = _Track(N, .75, kv)
    mem = np.zeros(Bv, bool)
    with torch.no_grad():
        for c in range(C):
            lens = plan[c]
            nd = [bool(L > 0 and not m) for L, m in zip(lens, mem)]
            ya = a.step(ks[c], qs[c], us[c], new_doc=nd, lengths=lens)
            yb = b.step_overlapped(ks[c], qs[c], us[c], new_doc=nd, lengths=lens,
                                   k_next=ks[c + 1] if c + 1 < C else None,
                                   next_lengths=plan[c + 1] if c + 1 < C else None)
            assert torch.equal(ya, yb), c
            assert torch.equal(a.B_past, b.B_past), c
            assert torch.equal(a.last["KV"], b.last["KV"]), c
            kc, qc, uc = ks[c].cpu(), qs[c].cpu(), us[c].cpu()
            for v in sample:
                if lens[v]:
                    tr.check(a, v, v, kc, qc, uc, lens[v], nd[v], ya)
            mem |= np.asarray(lens) > 0
    tr.assert_ok()


# --------------------------------------------------------------------------- prefetch bookkeeping
def test_prefetch_with_other_lengths_is_pooled_again(dev):
    Bv, Lmax = 3, 8
    a, _ = _engine(dev, 64)
    b, _ = _engine(dev, 64)
    g = torch.Generator().manual_seed(31)
    with torch.no_grad():
        k, q, _u = (t.to(dev) for t in _chunk(g, Bv, Lmax))
        a.prefetch(k, QN, lengths=[8, 8, 8])
        ya = a.step(k, q, new_doc=True, lengths=[8, 3, 5])          # other lengths: pooled again
        yb = b.step(k, q, new_doc=True, lengths=[8, 3, 5])
        assert torch.equal(ya, yb)
        k2, q2, u2 = (t.to(dev) for t in _chunk(g, Bv, Lmax))
        a.prefetch(k2, QN, lengths=[4, 0, 6])
        assert any(e["lens"] == (4, 0, 6) for e in a._pref)
        ya = a.step(k2, q2, u2, lengths=[4, 0, 6])                   # same lengths: the prefetch is consumed
        assert not any(e["lens"] == (4, 0, 6) for e in a._pref)
        yb = b.step(k2, q2, u2, lengths=[4, 0, 6])
        assert torch.equal(ya, yb)


# --------------------------------------------------------------------------- consolidate_video, per-video chunk counts
def test_consolidate_video_per_video_chunks(dev):
    from infinite_video_b200.video import consolidate_video
    Bv, Lmax, C = 3, 8, 4
    lengths = [[8, 8, 8], [8, 5, 8], [3, 0, 8], [0, 0, 2]]           # chunk counts 3, 2, 4
    eng, kv = _engine(dev, 64)
    g = torch.Generator().manual_seed(37)
    ks, qs, us = [], [], []
    for c in range(C):
        k, q, u = _chunk(g, Bv, Lmax, lens=lengths[c], fill=float("nan"))
        ks.append(k)
        qs.append(q)
        us.append(u)
    with torch.no_grad():
        mean = consolidate_video([eng], [k.to(dev) for k in ks], [[q.to(dev) for q in qs]],
                                 [[u.to(dev) for u in us]], reduce="mean", lengths=lengths)[0]
        eng.reset()
        per = consolidate_video([eng], [k.to(dev) for k in ks], [[q.to(dev) for q in qs]],
                                [[u.to(dev) for u in us]], lengths=lengths)[0]
    for c in range(C):
        for v in range(Bv):
            if lengths[c][v] == 0:
                assert not per[c][v].any()
    for v in range(Bv):
        orc = _oracle(64, .75, kv)
        acc, n = 0, 0
        for c in range(C):
            Lv = lengths[c][v]
            if Lv == 0:
                continue
            b_got = None                                  # draws of the engine's own run (ties would diverge)
            acc = acc + orc.forward(ks[c][v:v + 1, :Lv * 32], qs[c][v:v + 1], n == 0,
                                    us[c][v:v + 1] if n else None, b_override=b_got)
            n += 1
        assert relerr(mean[v:v + 1], acc / n) < TOL_CTX, v


# --------------------------------------------------------------------------- errors
def test_errors(dev):
    Bv, Lmax = 3, 8
    eng, _ = _engine(dev, 64)
    g = torch.Generator().manual_seed(41)
    k, q, u = (t.to(dev) for t in _chunk(g, Bv, Lmax))
    for bad in ([1, 8, 8], [9, 8, 8], [-2, 8, 8], [8, 8], torch.tensor([8, 8, 8], device=dev)):
        with pytest.raises(ValueError):
            eng.step(k, q, new_doc=True, lengths=bad)
    with pytest.raises(ValueError):
        eng.pool(k, lengths=[8, 1, 8])
    with torch.no_grad():
        eng.step(k, q, new_doc=[True, False, True], lengths=[8, 0, 8])      # slot 1 never received a chunk
        with pytest.raises(ValueError):
            eng.step(k, q, u, lengths=[8, 8, 8])
        eng.step(k, q, u, new_doc=[False, True, False], lengths=[8, 8, 8])
        eng.step(k, q, u, new_doc=[False, True, False], lengths=[8, 0, 8])   # clears slot 1
        with pytest.raises(ValueError):
            eng.step(k, q, u, lengths=[8, 4, 8])
        with pytest.raises(ValueError):
            eng.step(k, q, u)                                               # lock-step continue of an empty slot
        with pytest.raises(RuntimeError):
            eng.x_past()


def test_video_block_is_refused(dev):
    """The step in blocks of videos was removed: a non-zero `video_block` set on the engine is an error, not a no-op."""
    eng, _ = _engine(dev, 64)
    k, q, _u = (t.to(dev) for t in _chunk(torch.Generator().manual_seed(43), 3, 8))
    eng.video_block = 2
    with torch.no_grad():
        for run in (lambda: eng.step(k, q, new_doc=True), lambda: eng.step_overlapped(k, q, new_doc=True),
                    lambda: eng.step(k, q, new_doc=True, lengths=[8, 8, 8])):
            with pytest.raises(ValueError, match="video_block"):
                run()
        eng.video_block = 0
        assert bool(torch.isfinite(eng.step(k, q, new_doc=True)).all())
