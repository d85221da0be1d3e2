"""Ragged batches of variant R on the GPU: what per-video chunk lengths cost against the lock-step step, and what they
save against one engine per video.  Prints one JSON line per measurement and a summary line with the card.

  (a) bench shape (128 videos x 256 frames, N = 256), all lengths equal: ragged step_overlapped against lock-step
      step_overlapped with bin_pool on and off, alternating in one run;
  (b) lengths uniform over [2, 256] plus 10 % idle: chunks/s and HBM bandwidth on the bytes the step needs
      (4 * sum(L_v) * T * e pooled + state), against one Bv = 1 engine per video;
  (c) idle slots: the same padded batch with 0 / 10 / 50 % of the videos idle.

Each configuration cycles over 3 chunks of 3.2 GB (larger than the 126 MB L2), is warmed up on every shape first and
timed with CUDA events over `--steps` steps."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from infinite_video_b200.batched import BatchedRectLTM  # noqa: E402

T, E, QN, S = 32, 768, 32, 512


def card():
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                                      text=True).strip().splitlines()[0]
    except Exception as exc:                                # noqa: BLE001
        out = f"unknown ({exc})"
    return out


def engine(N, dev, **kw):
    torch.manual_seed(0)
    key, val = torch.nn.Linear(E, 768), torch.nn.Linear(E, 768)
    return BatchedRectLTM(N, .75, key.weight.detach(), key.bias.detach(), val.weight.detach(), val.bias.detach(),
                          device=dev, **kw)


def state_bytes(Bv, N, Q):
    # coefficients read + written, fp16 K|V read + written, queries and ctx, uniforms
    return Bv * (2 * N * E * 4 + 2 * N * 2 * 768 * 2 + 2 * Q * 768 * 4 + S * 8)


def run_overlapped(eng, ks, qs, us, lens_plan, steps, warmup):
    """Step the engine in a loop over the chunks; returns ms per step (events around `steps` steps)."""
    C = len(ks)
    n = steps + warmup
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    mem = None
    for i in range(n):
        c = i % C
        lens = lens_plan[i % len(lens_plan)] if lens_plan else None
        nl = lens_plan[(i + 1) % len(lens_plan)] if lens_plan else None
        if i == warmup:
            t0.record()
        if lens is None:
            eng.step_overlapped(ks[c], qs[c], us[c] if i else None, new_doc=(i == 0), k_next=ks[(c + 1) % C])
        else:
            present = np.asarray(lens) > 0
            if mem is None:
                mem = np.zeros(len(lens), bool)
            nd = [bool(p and not m) for p, m in zip(present, mem)]
            eng.step_overlapped(ks[c], qs[c], us[c], new_doc=nd, k_next=ks[(c + 1) % C], lengths=lens,
                                next_lengths=nl)
            mem |= present
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=6)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--videos", type=int, default=128)
    ap.add_argument("--frames", type=int, default=256)
    ap.add_argument("--num-basis", type=int, default=256)
    ap.add_argument("--out", default=None, help="also write the results as JSON to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("ragged_bench needs a CUDA device")
    dev = torch.device("cuda:0")
    Bv, L, N = args.videos, args.frames, args.num_basis
    g = torch.Generator(device=dev).manual_seed(1)
    ks = [torch.randn(Bv, L * T, E, device=dev, generator=g) for _ in range(3)]
    qs = [torch.randn(Bv, QN, 768, device=dev, generator=g) for _ in range(3)]
    us = [torch.rand(Bv, S, dtype=torch.float64, device=dev, generator=g) for _ in range(3)]
    rs = np.random.RandomState(2)
    results = {"card": card(), "shape": dict(videos=Bv, frames=L, num_basis=N, tokens=T, width=E)}

    # (a) equal lengths
    engs = {"lockstep_binpool": engine(N, dev), "lockstep_nobinpool": engine(N, dev, bin_pool=False),
            "ragged_equal": engine(N, dev)}
    plans = {"lockstep_binpool": None, "lockstep_nobinpool": None, "ragged_equal": [[L] * Bv]}
    for name in engs:
        run_overlapped(engs[name], ks, qs, us, plans[name], 2, args.warmup)
    a = {n: [] for n in engs}
    for _ in range(args.rounds):
        for name, eng in engs.items():
            eng.reset()
            a[name].append(run_overlapped(eng, ks, qs, us, plans[name], args.steps, args.warmup))
    pooled = 4 * Bv * L * T * E
    results["a"] = {n: dict(ms=[round(x, 4) for x in v], chunks_per_s=round(Bv / (min(v) / 1e3)),
                            GBps=round((pooled + state_bytes(Bv, N, QN)) / (min(v) / 1e3) / 1e9, 1))
                    for n, v in a.items()}
    del engs

    # (b) lengths uniform over [2, L] + 10 % idle, against one engine per video
    plan = []
    for _ in range(6):
        lens = rs.randint(2, L + 1, size=Bv)
        lens[rs.rand(Bv) < 0.1] = 0
        plan.append([int(x) for x in lens])
    eng = engine(N, dev)
    run_overlapped(eng, ks, qs, us, plan, 2, args.warmup)
    rb = []
    for _ in range(args.rounds):
        eng.reset()
        rb.append(run_overlapped(eng, ks, qs, us, plan, args.steps, args.warmup))
    present = float(np.mean([sum(1 for x in p if x) for p in plan]))
    frames = float(np.mean([sum(p) for p in plan]))
    need = 4 * frames * T * E + state_bytes(Bv, N, QN)
    results["b_ragged"] = dict(ms=[round(x, 4) for x in rb], chunks_per_s=round(present / (min(rb) / 1e3)),
                               GBps_needed=round(need / (min(rb) / 1e3) / 1e9, 1), mean_frames=frames,
                               mean_present=present)
    del eng
    # one Bv = 1 engine per video (sequential steps of the same chunks, each with its own length)
    singles = [engine(N, dev) for _ in range(Bv)]
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    steps1 = max(3, args.steps // 5)
    times = []
    for r in range(args.rounds + 1):
        started = [False] * Bv
        for i in range(steps1 + 2):
            if i == 2:
                t0.record()
            c, lens = i % 3, plan[i % len(plan)]
            for v in range(Bv):
                if lens[v] == 0:
                    continue
                k = ks[c][v:v + 1, :lens[v] * T]
                singles[v].step(k, qs[c][v:v + 1], us[c][v:v + 1] if started[v] else None, new_doc=not started[v])
                started[v] = True
        t1.record()
        torch.cuda.synchronize()
        if r:
            times.append(t0.elapsed_time(t1) / steps1)
    results["b_per_video_engines"] = dict(ms=[round(x, 4) for x in times],
                                          chunks_per_s=round(present / (min(times) / 1e3)))
    del singles

    # (c) idle slots: all videos at L frames, a share of them idle
    eng = engine(N, dev)
    c_res = {}
    for share in (0.0, 0.1, 0.5):
        lens = [0 if (v % 10) < share * 10 else L for v in range(Bv)]
        plan_c = [lens]
        run_overlapped(eng, ks, qs, us, plan_c, 2, args.warmup)
        ts = []
        for _ in range(args.rounds):
            eng.reset()
            ts.append(run_overlapped(eng, ks, qs, us, plan_c, args.steps, args.warmup))
        n_present = sum(1 for x in lens if x)
        c_res[f"idle_{int(share * 100)}pct"] = dict(ms=[round(x, 4) for x in ts], present=n_present,
                                                    us_per_present_chunk=round(min(ts) * 1e3 / n_present, 3))
    results["c"] = c_res
    print(json.dumps(results))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(results, f, indent=1)


if __name__ == "__main__":
    main()
