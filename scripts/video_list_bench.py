"""Per-video chunk tensors against a padded batch, on the GPU: what the copy into a padded chunk costs a serving loop,
and what stepping the LTM on the per-video tensors directly (`step_overlapped(k=[...], chunk_frames=L)`) gives back.

Three arms, interleaved in one run at the bench shape (128 videos x 256 frames x 32 tokens x 768, N = 256), for fp32
and fp16 chunks, with all lengths 256 and with lengths uniform over [2, 256] plus 10 % idle videos:
  (i)   padded: the chunks sit in padded [Bv, L*T, e] tensors already, ragged step -- no assembly at all;
  (ii)  assemble: the chunks sit in per-video tensors and every step first copies them into a fresh padded chunk
        (`torch.empty` + one copy per video, the loop of INTEGRATION.md section 3), then the ragged step;
  (iii) list: the same per-video tensors handed over as a list, each frame pooled where it lives.
Each arm cycles over 3 chunks (2-3 GB each in fp32, well above the 126 MB L2); every round runs `--steps`
`step_overlapped` steps per arm after `--warmup` steps, timed with CUDA events; the best of `--rounds` rounds is kept.
Host enqueue time is a host clock around the loop body (assembly and step call), without a synchronise.  Also the
pooling kernel alone, pointer table against padded ragged chunk, on the same frames.  Prints one JSON line per
configuration and a summary line with the card's name and power limit."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from infinite_video_b200 import ops  # noqa: E402
from infinite_video_b200.batched import BatchedRectLTM  # noqa: E402

T, E, QN, S = 32, 768, 32, 512
ARMS = ("padded", "assemble", "list")


def card():
    try:
        return subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                                       text=True).strip().splitlines()[0]
    except Exception as exc:                                # noqa: BLE001
        return f"unknown ({exc})"


def engine(N, dev):
    torch.manual_seed(0)
    key, val = torch.nn.Linear(E, 768), torch.nn.Linear(E, 768)
    return BatchedRectLTM(N, .75, key.weight.detach(), key.bias.detach(), val.weight.detach(), val.bias.detach(),
                          device=dev)


def state_bytes(Bv, N, Q):
    # coefficients read + written, fp16 K|V read + written, queries and ctx, uniforms
    return Bv * (2 * N * E * 4 + 2 * N * 2 * 768 * 2 + 2 * Q * 768 * 4 + S * 8)


def assemble(parts, L, dtype, dev):
    """What a serving loop does without the list form: a padded chunk, one copy per video."""
    k = torch.empty(len(parts), L * T, E, device=dev, dtype=dtype)
    for v, p in enumerate(parts):
        if p is not None:
            k[v, :p.shape[0]] = p
    return k


def run(eng, arm, data, steps, warmup):
    """`steps` overlapped steps after `warmup`; returns (ms per step on the device, host ms per step, last ctx)."""
    plan, parts, padded, qs, us, L = data["plan"], data["parts"], data["padded"], data["qs"], data["us"], data["L"]
    C, Bv = len(plan), len(plan[0])
    eng.reset()
    mem = np.zeros(Bv, bool)
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def chunk(c):
        if arm == "padded":
            return padded[c]
        if arm == "assemble":
            return assemble(parts[c], L, padded[c].dtype, padded[c].device)
        return parts[c]

    host = 0.0
    cur = chunk(0)
    for i in range(warmup + steps):
        if i == warmup:
            torch.cuda.synchronize()
            t0.record()
            host = 0.0
        c, n = i % C, (i + 1) % C
        lens = plan[c]
        present = np.asarray(lens) > 0
        nd = [bool(p and not m) for p, m in zip(present, mem)]
        h = time.perf_counter()
        nxt = chunk(n)
        if arm == "list":
            y = eng.step_overlapped(cur, qs[c], us[c], new_doc=nd, k_next=nxt, chunk_frames=L)
        else:
            y = eng.step_overlapped(cur, qs[c], us[c], new_doc=nd, k_next=nxt, lengths=lens, next_lengths=plan[n])
        host += time.perf_counter() - h
        cur = nxt
        mem |= present
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1) / steps, host * 1e3 / steps, y


def pool_kernels(data, reps, rounds):
    """The pooling kernel alone on the frames of each chunk: pointer table against the padded ragged chunk."""
    plan, parts, padded, L = data["plan"], data["parts"], data["padded"], data["L"]
    eng = data["eng"]
    best = {"ptrs": [], "ragged": []}
    nbytes = 0
    setups = []
    for c in range(len(plan)):
        lens, frames = plan[c], sum(plan[c])
        _, offs, table = eng._lengths_dev(lens, [0 if p is None else p.data_ptr() for p in parts[c]])
        out = torch.empty(frames, 1, E, device=padded[c].device)
        code = ops.CHUNK_DTYPES[padded[c].dtype]
        setups.append((lens, frames, offs, table, out, code))
        nbytes += frames * T * E * padded[c].element_size() + frames * E * 4
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(rounds):
        for kind in best:
            torch.cuda.synchronize()
            t0.record()
            for _ in range(reps):
                for c, (lens, frames, offs, table, out, code) in enumerate(setups):
                    if kind == "ptrs":
                        ops.pool_ptrs(table, code, out, offs, len(lens), L, T, E, 1, frames)
                    else:
                        ops.pool_into(padded[c], out, L, T, 1, offs=offs, frames=frames)
            t1.record()
            torch.cuda.synchronize()
            best[kind].append(t0.elapsed_time(t1) / reps)
    return {k: dict(ms_per_3_chunks=round(min(v), 4), GBps=round(nbytes / (min(v) / 1e3) / 1e9, 1))
            for k, v in best.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=6)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--videos", type=int, default=128)
    ap.add_argument("--frames", type=int, default=256)
    ap.add_argument("--num-basis", type=int, default=256)
    ap.add_argument("--dtypes", default="fp32,fp16")
    ap.add_argument("--out", default=None, help="also write the results as JSON to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("video_list_bench needs a CUDA device")
    dev = torch.device("cuda:0")
    Bv, L, N = args.videos, args.frames, args.num_basis
    results = {"card": card(), "shape": dict(videos=Bv, frames=L, num_basis=N, tokens=T, width=E), "runs": []}
    rs = np.random.RandomState(2)
    for dname in args.dtypes.split(","):
        dtype = {"fp32": torch.float32, "fp16": torch.float16}[dname]
        for mode in ("all", "uniform"):
            plan = []
            for _ in range(3):
                if mode == "all":
                    plan.append([L] * Bv)
                else:
                    lens = rs.randint(2, L + 1, size=Bv)
                    lens[rs.rand(Bv) < 0.1] = 0
                    plan.append([int(x) for x in lens])
            g = torch.Generator(device=dev).manual_seed(1)
            parts = [[torch.randn(n * T, E, device=dev, generator=g).to(dtype) if n else None for n in lens]
                     for lens in plan]
            padded = [assemble(p, L, dtype, dev) for p in parts]
            qs = [torch.randn(Bv, QN, 768, device=dev, generator=g) for _ in range(3)]
            us = [torch.rand(Bv, S, dtype=torch.float64, device=dev, generator=g) for _ in range(3)]
            engs = {a: engine(N, dev) for a in ARMS}
            data = dict(plan=plan, parts=parts, padded=padded, qs=qs, us=us, L=L, eng=engs["list"])
            for a in ARMS:
                run(engs[a], a, data, 2, args.warmup)
            dev_ms, host_ms, last = {a: [] for a in ARMS}, {a: [] for a in ARMS}, {}
            for _ in range(args.rounds):
                for a in ARMS:
                    d, h, y = run(engs[a], a, data, args.steps, args.warmup)
                    dev_ms[a].append(d)
                    host_ms[a].append(h)
                    last[a] = y
            same = all(torch.equal(last[a], last["padded"]) for a in ARMS)
            present = float(np.mean([sum(1 for x in p if x) for p in plan]))
            frames = float(np.mean([sum(p) for p in plan]))
            need = frames * T * E * padded[0].element_size() + state_bytes(Bv, N, QN)
            res = dict(dtype=dname, lengths=mode, mean_frames=frames, mean_present=present, same_ctx=same,
                       bytes_needed_per_step=int(need))
            for a in ARMS:
                best = min(dev_ms[a])
                res[a] = dict(ms=[round(x, 4) for x in dev_ms[a]], present_chunks_per_s=round(present / (best / 1e3)),
                              GBps_needed=round(need / (best / 1e3) / 1e9, 1),
                              host_enqueue_ms=round(min(host_ms[a]), 4))
            res["pool_kernel"] = pool_kernels(data, 10, args.rounds)
            print(json.dumps(res), flush=True)
            results["runs"].append(res)
            del engs, data, parts, padded
            torch.cuda.empty_cache()
    print(json.dumps({"card": results["card"], "shape": results["shape"]}))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(results, f, indent=1)


if __name__ == "__main__":
    main()
