#!/usr/bin/env python
"""Chunk-calls/s of the caller's cross-attention branch (`CrossAttentionLTM.forward`) on a batch of videos, lock-step
against ragged (`lengths=`), at Video-LLaMA widths: e = D = 768, H = 12, Q = 32, T = 32, L = 256, num_basis 256.

  (i)   lock-step: every video a full chunk of L frames, no lengths
  (ii)  ragged, every length = L
  (iii) ragged, lengths uniform in [2, L] with 10 % of the videos idle; rate = PRESENT video chunk-calls/s

Each case is timed with CUDA events over --iters calls after --warmup calls (alternating between two chunk tensors,
so that the shared pooling slot never hands a call the previous call's frames), for the whole branch and for the
short-term half alone.  The short-term FLOPs and bytes each case needs are computed from the lengths (only the two
large contractions, the row softmax and the pool + fp16 pass).  Prints one JSON object; the card's name and power
limit are read in the same run.

  python scripts/ragged_cross_attention_bench.py [--videos 32] [--iters 20] [--warmup 5] [--out FILE]
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

E, D, H, Q, T, L, NB = 768, 768, 12, 32, 32, 256, 256


def card():
    name = torch.cuda.get_device_name(0)
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(torch.cuda.current_device())
        limit = pynvml.nvmlDeviceGetPowerManagementLimit(h) / 1000.0
    except Exception as exc:                          # the number stays unlabelled rather than guessed
        limit = f"unavailable ({type(exc).__name__})"
    return name, limit


def short_term_cost(lens):
    """FLOPs and HBM bytes of the short-term half for these lengths (frames per video): the score and value GEMMs
    (2 x 2 H Q e n_v), the chunk read once as fp32 and written as fp16, k16 read by both GEMMs, S written and read,
    P written and read."""
    n = np.asarray(lens, np.float64) * T
    flops = float((4 * H * Q * E * n).sum())
    byts = float((n * E * (4 + 2 + 2 * 2) + H * Q * n * (4 * 2 + 2 * 2)).sum())
    return flops, byts


def timed(fn, calls, warmup):
    for i in range(warmup):
        fn(i)
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for i in range(calls):
        fn(i)
    t1.record()
    t1.synchronize()
    return t0.elapsed_time(t1) / calls


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--videos", type=int, default=32)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("ragged_cross_attention_bench needs a CUDA device")
    from infinite_video_b200 import LongTermAttention
    from infinite_video_b200.cross_attention import CrossAttentionLTM
    dev = torch.device("cuda:0")
    B = a.videos
    torch.manual_seed(0)
    lq, lk, lv = (torch.nn.Linear(E, D).to(dev) for _ in range(3))
    rs = np.random.RandomState(1)
    ragged = rs.randint(2, L + 1, size=B)
    ragged[rs.choice(B, max(1, round(0.1 * B)), replace=False)] = 0
    cases = {"lockstep": None, "ragged_full": [L] * B, "ragged_uniform": ragged.tolist()}
    g = torch.Generator(device=dev).manual_seed(2)
    encs = [torch.randn(B, L * T, E, device=dev, generator=g) for _ in range(2)]
    hidden = torch.randn(B, Q, D, device=dev, generator=g)
    u = torch.rand(B, 512, dtype=torch.float64)
    res = {}
    for name, lens in cases.items():
        m = CrossAttentionLTM(lq, lk, lv, 0.5, NB, .75, tokens_per_frame=T, videos_per_pass=B)
        m(hidden, encs[0], new_video=True, lengths=lens)                  # first chunk of every video
        LongTermAttention._shared_pool.update(key=None, x=None, k16=None)

        def call(i, m=m, lens=lens):
            m(hidden, encs[i % 2], new_video=False, u=u, lengths=lens)
        q = m._linear(hidden.reshape(B * Q, D), m.query, "tf32x3").view(B, Q, D)

        def stm(i, m=m, lens=lens):
            m.short_term(q, encs[i % 2], lengths=lens)
        ms = timed(call, a.iters, a.warmup)
        ms_stm = timed(stm, a.iters, a.warmup)
        present = B if lens is None else int(sum(1 for x in lens if x))
        flops, byts = short_term_cost([L] * B if lens is None else lens)
        res[name] = dict(ms_per_call=ms, present_chunk_calls_per_s=present / (ms * 1e-3), short_term_ms=ms_stm,
                         short_term_gflop=flops / 1e9, short_term_gbytes=byts / 1e9,
                         frames=int(L * B if lens is None else sum(lens)), present_videos=present)
    name, limit = card()
    out = dict(card=name, power_limit_w=limit, videos=B, L=L, T=T, e=E, H=H, Q=Q, num_basis=NB, iters=a.iters,
               warmup=a.warmup, cases=res)
    line = json.dumps(out)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
