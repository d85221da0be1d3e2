"""Bitwise digests of the variant-R step: one SHA-256 per (configuration, entry point) over the ctx of every chunk and,
after the last chunk, B_past, the projected memory (K|V, or V on the transposed-key path), the sticky histogram
partials and the last draws (idx, b).  Inputs are seeded; every entry point runs 4 chunks on a fresh engine.

A change that must not alter results (a refactor of the step) is checked by running this against the tree before and
after it, on the same GPU, and diffing the two outputs:

    python scripts/step_digest.py --root OLD_TREE --out old.txt
    python scripts/step_digest.py --root .        --out new.txt
    diff old.txt new.txt

Buffers the step writes only on some calls (the draws of a first or non-sticky chunk, the rows of a video that does not
continue its memory) are filled with a sentinel after the first chunk, so the digest never covers uninitialised
memory."""
import argparse
import hashlib
import os
import sys

CHUNKS = 4
SMALL = dict(Bv=3, L=8, N=64)
BIG = dict(Bv=128, L=256, N=256)         # production shape: per-bin pooling (bin_pool=None), 256-wide GEMM tiles

LOCKSTEP = ("step", "pool+step", "prefetch+step", "overlapped", "host")
RAGGED = ("ragged_step", "ragged_overlapped", "ragged_pool+step")

# name, engine keyword arguments, shape, chunk dtype, entry points
CONFIGS = [
    ("default", {}, SMALL, "fp32", LOCKSTEP + RAGGED),
    ("production", {}, BIG, "fp32", LOCKSTEP[:4] + RAGGED),
    ("kv_fp32", dict(kv_dtype="fp32"), SMALL, "fp32", LOCKSTEP + RAGGED),
    ("proj_fp32", dict(proj_operands="fp32"), SMALL, "fp32", LOCKSTEP),
    ("proj_fp32_kv_fp32", dict(proj_operands="fp32", kv_dtype="fp32"), SMALL, "fp32", LOCKSTEP + RAGGED),
    ("no_kv_state", dict(kv_state=False), SMALL, "fp32", LOCKSTEP + RAGGED),
    ("tf32x3", dict(precision="tf32x3"), SMALL, "fp32", LOCKSTEP + RAGGED),
    ("tf32x3_proj_tf32", dict(precision="tf32x3", proj_precision="tf32"), SMALL, "fp32", LOCKSTEP),
    ("generic", dict(fast_attn=False), SMALL, "fp32", LOCKSTEP + RAGGED),
    ("generic_proj_tf32x3", dict(fast_attn=False, proj_precision="tf32x3"), SMALL, "fp32", LOCKSTEP),
    ("generic_no_kv_state_proj_tf32x3", dict(fast_attn=False, kv_state=False, proj_precision="tf32x3"), SMALL, "fp32",
     LOCKSTEP),
    ("n512", {}, dict(Bv=2, L=32, N=512), "fp32", LOCKSTEP + RAGGED),
    ("bin_pool_true", dict(bin_pool=True), dict(Bv=2, L=256, N=256), "fp32", LOCKSTEP),
    ("bin_pool_false", dict(bin_pool=False), dict(Bv=2, L=256, N=256), "fp32", LOCKSTEP),
    ("not_sticky", dict(sticky=False), SMALL, "fp32", LOCKSTEP + RAGGED),
    ("mixed_new_doc", {}, SMALL, "fp32", LOCKSTEP),
    ("mixed_new_doc_bins", dict(bin_pool=True), dict(Bv=2, L=256, N=256), "fp32", LOCKSTEP),   # stale per-bin prefetch
    # 16-bit chunks: every entry point must print the digest of `step` on the same chunks
    ("fp16_chunk", {}, SMALL, "fp16", LOCKSTEP + ("ragged_step", "ragged_pool+step", "ragged_overlapped")),
    ("bf16_chunk", {}, SMALL, "bf16", LOCKSTEP + ("ragged_step", "ragged_pool+step", "ragged_overlapped")),
    ("production_fp16", {}, BIG, "fp16", LOCKSTEP[:4] + RAGGED),
    # num_basis 512 with K|V on the tf32 grid: the fp32 two-half attention (ltm_cont_attn_rect_tc_split)
    ("n512_kv_fp32", dict(kv_dtype="fp32"), dict(Bv=2, L=32, N=512), "fp32", LOCKSTEP + RAGGED),
]


def _inputs(torch, dev, cfg, shape, dtype, S, seed):
    Bv, L = shape["Bv"], shape["L"]
    g = torch.Generator(device=dev).manual_seed(seed)
    dt = dict(fp32=torch.float32, fp16=torch.float16, bf16=torch.bfloat16)[dtype]
    ks = [torch.randn(Bv, L * 32, 768, generator=g, device=dev).to(dt) for _ in range(CHUNKS)]
    qs = [torch.randn(Bv, 32, 768, generator=g, device=dev) for _ in range(CHUNKS)]
    us = [torch.rand(Bv, S, generator=g, device=dev, dtype=torch.float64) for _ in range(CHUNKS)]
    # lock-step new_doc: a first chunk, then continuations; `mixed_new_doc` restarts every other video at chunk 2
    nds = [True] + [False] * (CHUNKS - 1)
    if cfg.startswith("mixed_new_doc"):
        nds[2] = [v % 2 == 0 for v in range(Bv)]
    return ks, qs, us, nds


def _ragged_schedule(np, Bv, L, seed):
    """Per-chunk lengths (0 = idle) and host new_doc flags: idle slots, slots without memory that start a document,
    and a document restarted in the middle."""
    rng = np.random.RandomState(seed)
    mem = np.zeros(Bv, bool)
    lens, nds = [], []
    for c in range(CHUNKS):
        ln = rng.randint(2, L + 1, Bv)
        ln[rng.rand(Bv) < 0.15] = 0
        ln[L % Bv] = L                               # one full-length video
        if c in (0, 1, 3):
            ln[c % Bv] = 0                           # idle (a cleared, empty slot at chunk 0)
        nd = np.ones(Bv, bool) if c == 0 else rng.rand(Bv) < 0.1
        if c == 2:
            nd[(c + 1) % Bv] = True
        nd |= (ln > 0) & ~mem
        mem = np.where(nd, ln > 0, mem)
        lens.append(ln.tolist())
        nds.append(nd.tolist())
    return lens, nds


def _run(torch, eng, entry, ks, qs, us, nds, rag):
    Q = qs[0].shape[1]
    ctxs = []
    host = entry == "host"
    if host:
        ks = [k.cpu().pin_memory() for k in ks]
        qs = [q.cpu().pin_memory() for q in qs]
        us = [u.cpu().pin_memory() for u in us]
    if rag is not None:
        lens, rnds = rag
    for c in range(CHUNKS):
        k, q = ks[c], qs[c]
        u = us[c] if c else None
        nd = nds[c]
        if not host and isinstance(nd, list):
            nd = torch.tensor(nd, device=k.device)          # device flags: the lock-step step takes them as they are
        nxt = c + 1 < CHUNKS
        if entry == "step":
            ctx = eng.step(k, q, u, new_doc=nd)
        elif entry == "pool+step":
            ctx = eng.step(k, q, u, new_doc=nd, pooled=eng.pool(k))
        elif entry == "prefetch+step":
            if c == 0:
                eng.prefetch(k, Q)
            if nxt:
                eng.prefetch(ks[c + 1], Q, update=True)     # a continuation is expected (mixed flags: pooled again)
            ctx = eng.step(k, q, u, new_doc=nd)
        elif entry == "overlapped":
            ctx = eng.step_overlapped(k, q, u, new_doc=nd, k_next=ks[c + 1] if nxt else None)
        elif entry == "host":
            ctx = eng.step_host(k, q, u, new_doc=nd)
            torch.cuda.synchronize()
        elif entry == "ragged_step":
            ctx = eng.step(k, q, us[c], new_doc=rnds[c], lengths=lens[c])
        elif entry == "ragged_overlapped":
            ctx = eng.step_overlapped(k, q, us[c], new_doc=rnds[c], lengths=lens[c], k_next=ks[c + 1] if nxt else None,
                                      next_lengths=lens[c + 1] if nxt else None)
        elif entry == "ragged_pool+step":
            ctx = eng.step(k, q, us[c], new_doc=rnds[c], pooled=eng.pool(k, lengths=lens[c]), lengths=lens[c])
        else:
            raise ValueError(entry)
        ctxs.append(ctx.clone())
        if c == 0:
            eng.last["idx"].fill_(-7)
            eng.last["b"].fill_(-7)
    torch.cuda.synchronize()
    h = hashlib.sha256()
    last = eng.last
    kv = last["KV"] if last["KV"] is not None else last["V"]
    for t in ctxs + [eng.B_past, kv, eng._hist, last["idx"], last["b"]]:
        h.update(b"none" if t is None else t.detach().contiguous().cpu().numpy().tobytes())
    return h.hexdigest()


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--root", required=True, help="tree whose infinite_video_b200 package is imported")
    ap.add_argument("--out", required=True, help="file that receives one 'config entry sha256' line per run")
    ap.add_argument("--only", default=None, help="comma-separated configuration names (default: all)")
    args = ap.parse_args()
    root = os.path.abspath(args.root)
    sys.path.insert(0, root)
    import numpy as np
    import torch
    import infinite_video_b200
    from infinite_video_b200.batched import BatchedRectLTM
    assert os.path.dirname(os.path.abspath(infinite_video_b200.__file__)) == os.path.join(root, "infinite_video_b200")

    dev = torch.device("cuda", 0)
    g = torch.Generator().manual_seed(7)
    w = (torch.randn(768, 768, generator=g) * 0.03, torch.randn(768, generator=g) * 0.1,
         torch.randn(768, 768, generator=g) * 0.03, torch.randn(768, generator=g) * 0.1)
    only = set(args.only.split(",")) if args.only else None
    lines = []
    with torch.no_grad():
        for i, (name, kw, shape, dtype, entries) in enumerate(CONFIGS):
            if only is not None and name not in only:
                continue
            ks = qs = us = None
            for entry in entries:
                eng = BatchedRectLTM(shape["N"], 0.75, *w, device=dev, **kw)
                if ks is None:
                    ks, qs, us, nds = _inputs(torch, dev, name, shape, dtype, eng.S, 100 + i)
                rag = _ragged_schedule(np, shape["Bv"], shape["L"], 200 + i) if entry.startswith("ragged") else None
                line = f"{name} {entry} {_run(torch, eng, entry, ks, qs, us, nds, rag)}"
                print(line, flush=True)
                lines.append(line)
                del eng
            del ks, qs, us
            torch.cuda.empty_cache()
    with open(args.out, "w") as f:
        f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
