"""16-bit chunks through the overlapped step on one B200: what fp16 / bfloat16 encoder states buy against fp32 ones.
Prints one JSON object (and writes it to --out).

  (a) step_overlapped at the NExT-QA shape (128 videos x 256 frames x 32 x 768, num_basis 256) and at cfg3, the
      VideoChat2 shape (64 videos x 16 frames x 196 x 1024, num_basis 64), with fp32, fp16 and bf16 chunks.  16-bit
      chunks run with the grid bound of the K/V projection beside the pooling (`gemm_ctas_overlap`) on and off.  The
      arms alternate inside each round; the best of `--rounds` rounds is reported.  Each arm cycles over 3 chunks
      (0.8 - 3.2 GB each, larger than the 126 MB L2; no flush).  Reported: chunks/s, pooled bytes/s (chunk bytes over
      step time), and the step's algorithmic bytes over step time against the 7.7 TB/s HBM3e data-sheet peak.
  (b) step_host at the NExT-QA shape with pinned fp32 and fp16 host chunks (PCIe-bound: the copy halves).
  (c) parity at the NExT-QA shape: 4 videos x 4 chunks of fp16 through step_overlapped against the oracle run on the
      up-cast chunks (flips / draws, coefficient and ctx error, no guard band).

The card name and power limit are read in the same run."""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from infinite_video_b200.batched import BatchedRectLTM  # noqa: E402

QN, S, D = 32, 512, 768
HBM_PEAK = 7.7e12                  # B/s, HBM3e data sheet of one HGX B200 GPU
SHAPES = {"nextqa": dict(Bv=128, L=256, T=32, e=768, N=256, Q=32),
          "cfg3": dict(Bv=64, L=16, T=196, e=1024, N=64, Q=96)}
DTYPES = {"fp32": torch.float32, "fp16": torch.float16, "bf16": torch.bfloat16}


def card():
    try:
        return subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm",
                                        "--format=csv,noheader"], text=True).strip().splitlines()[0]
    except Exception as exc:                                # noqa: BLE001
        return f"unknown ({exc})"


def engine(sh, dev, **kw):
    torch.manual_seed(0)
    key, val = torch.nn.Linear(sh["e"], D), torch.nn.Linear(sh["e"], D)
    return BatchedRectLTM(sh["N"], .75, key.weight.detach(), key.bias.detach(), val.weight.detach(),
                          val.bias.detach(), tokens_per_frame=sh["T"], device=dev, **kw)


def step_bytes(sh, elem):
    """Algorithmic bytes of one call per video, SURVEY 8(d) with the chunk's element size:
    elem*L*T*e (read k) + 4*(2*Q*D + 2*N*e) (q, ctx, B_past, B) + 8*S (u)."""
    return elem * sh["L"] * sh["T"] * sh["e"] + 4 * (2 * sh["Q"] * D + 2 * sh["N"] * sh["e"]) + 8 * S


def run_overlapped(eng, ks, qs, us, steps, warmup):
    C = len(ks)
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    eng.reset()
    for i in range(warmup + steps):
        if i == warmup:
            t0.record()
        c = i % C
        eng.step_overlapped(ks[c], qs[c], us[c] if i else None, new_doc=(i == 0), k_next=ks[(c + 1) % C])
    t1.record()
    torch.cuda.synchronize()
    eng.cancel_prefetch()
    return t0.elapsed_time(t1) / steps


def overlapped_arms(name, sh, dev, args):
    Bv, LT, e = sh["Bv"], sh["L"] * sh["T"], sh["e"]
    g = torch.Generator(device=dev).manual_seed(1)
    qs = [torch.randn(Bv, sh["Q"], D, device=dev, generator=g) for _ in range(3)]
    us = [torch.rand(Bv, S, dtype=torch.float64, device=dev, generator=g) for _ in range(3)]
    chunks = {}
    for dn, dt in DTYPES.items():
        chunks[dn] = [torch.randn(Bv, LT, e, device=dev, generator=g).to(dt) for _ in range(3)]
    arms = {"fp32": ("fp32", True), "fp16_bound": ("fp16", True), "fp16_nobound": ("fp16", False),
            "bf16_bound": ("bf16", True), "bf16_nobound": ("bf16", False)}
    engs = {}
    for arm, (dn, bound) in arms.items():
        engs[arm] = engine(sh, dev)
        if not bound:
            engs[arm].gemm_ctas_overlap = 0
        run_overlapped(engs[arm], chunks[dn], qs, us, 2, args.warmup)
    times = {arm: [] for arm in arms}
    for _ in range(args.rounds):
        for arm, (dn, _b) in arms.items():
            times[arm].append(run_overlapped(engs[arm], chunks[dn], qs, us, args.steps, args.warmup))
    out = {}
    for arm, (dn, bound) in arms.items():
        elem = 4 if dn == "fp32" else 2
        s = min(times[arm]) * 1e-3
        sb = step_bytes(sh, elem) * Bv
        out[arm] = dict(ms=[round(x, 4) for x in times[arm]], chunks_per_s=round(Bv / s),
                        pooled_GBps=round(elem * Bv * LT * e / s / 1e9, 1),
                        step_GBps=round(sb / s / 1e9, 1), roofline_frac=round(sb / s / HBM_PEAK, 4),
                        algorithmic_bytes_per_step=sb, projection_bound=bound,
                        gemm_ctas=engs[arm].gemm_ctas_overlap if bound else 0)
    del engs, chunks
    torch.cuda.empty_cache()
    return out


def host_arms(sh, dev, args):
    Bv, LT, e = sh["Bv"], sh["L"] * sh["T"], sh["e"]
    g = torch.Generator().manual_seed(2)
    qs = [torch.randn(Bv, sh["Q"], D, generator=g).pin_memory() for _ in range(2)]
    us = [torch.rand(Bv, S, dtype=torch.float64, generator=g).pin_memory() for _ in range(2)]
    out = {}
    engs, chunks = {}, {}
    for dn in ("fp32", "fp16"):
        chunks[dn] = [torch.randn(Bv, LT, e, generator=g).to(DTYPES[dn]).pin_memory() for _ in range(2)]
        engs[dn] = engine(sh, dev)
    times = {dn: [] for dn in engs}
    for r in range(args.rounds + 1):
        for dn, eng in engs.items():
            eng.reset()
            res = torch.empty(Bv, sh["Q"], D, pin_memory=True)
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            for i in range(args.host_steps + 1):
                if i == 1:
                    t0.record()
                eng.step_host(chunks[dn][i % 2], qs[i % 2], us[i % 2] if i else None, new_doc=(i == 0), out=res)
            t1.record()
            torch.cuda.synchronize()
            if r:                                           # round 0 warms up
                times[dn].append(t0.elapsed_time(t1) / args.host_steps)
    for dn in engs:
        elem = 4 if dn == "fp32" else 2
        s = min(times[dn]) * 1e-3
        h2d = elem * Bv * LT * e + 4 * Bv * sh["Q"] * D + 8 * Bv * S
        out[dn] = dict(ms=[round(x, 3) for x in times[dn]], chunks_per_s=round(Bv / s),
                       h2d_bytes_per_step=h2d, h2d_GBps=round(h2d / s / 1e9, 1))
    return out


def parity(dev, videos=4, chunks=4):
    from oracle import ltm_oracle as O
    sh = SHAPES["nextqa"]
    torch.manual_seed(0)
    key, val = torch.nn.Linear(sh["e"], D), torch.nn.Linear(sh["e"], D)
    w = (key.weight.detach(), key.bias.detach(), val.weight.detach(), val.bias.detach())
    orcs = [O.RectLTM(sh["N"], .75, *w, tokens_per_frame=sh["T"], rebuild_tables=False, faithful_quadrature=False)
            for _ in range(videos)]
    eng = BatchedRectLTM(sh["N"], .75, *w, tokens_per_frame=sh["T"], device=dev)
    g = torch.Generator().manual_seed(4321)
    ks = [torch.randn(videos, sh["L"] * sh["T"], sh["e"], generator=g).half() for _ in range(chunks)]
    rel = lambda a, b: float((a.double().cpu() - b.double()).abs().max() / b.double().abs().max())
    worst_ctx = worst_B = 0.0
    flips = draws = 0
    kd = [k.to(dev) for k in ks]
    with torch.no_grad():
        for c in range(chunks):
            q = torch.randn(videos, sh["Q"], D, generator=g)
            u = torch.rand(videos, S, dtype=torch.float64, generator=g)
            got = eng.step_overlapped(kd[c], q.to(dev), u.to(dev) if c else None, new_doc=(c == 0),
                                      k_next=kd[c + 1] if c + 1 < chunks else None)
            b_got = eng.last["b"].cpu().long() if c else None
            for v in range(videos):
                want = orcs[v].forward(ks[c][v:v + 1].float(), q[v:v + 1], c == 0, u[v:v + 1],
                                       b_override=b_got[v:v + 1] if c else None)
                worst_ctx = max(worst_ctx, rel(got[v:v + 1], want))
                worst_B = max(worst_B, rel(eng.B_past[v:v + 1], orcs[v].B_past))
                if c:
                    flips += int((orcs[v].last["b_own"] != b_got[v:v + 1]).sum())
                    draws += b_got[v:v + 1].numel()
    return dict(videos=videos, chunks=chunks, dtype="fp16", ctx_max_relerr=worst_ctx, coeff_max_relerr=worst_B,
                flips=flips, draws=draws, ok=bool(worst_ctx < 1e-3 and worst_B < 1e-5 and flips <= 0.01 * draws))


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=6)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--host-steps", type=int, default=4)
    ap.add_argument("--only", default=None, help="comma-separated parts: nextqa,cfg3,host,parity (default: all)")
    ap.add_argument("--out", default=None, help="also write the results as JSON to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("half_chunk_bench needs a CUDA device")
    dev = torch.device("cuda:0")
    parts = args.only.split(",") if args.only else ["nextqa", "cfg3", "host", "parity"]
    res = {"card": card(), "shapes": SHAPES, "hbm_peak_Bps": HBM_PEAK}
    for name in ("nextqa", "cfg3"):
        if name in parts:
            res[name] = overlapped_arms(name, SHAPES[name], dev, args)
            print(json.dumps({name: res[name]}), flush=True)
    if "host" in parts:
        res["host_nextqa"] = host_arms(SHAPES["nextqa"], dev, args)
        print(json.dumps({"host_nextqa": res["host_nextqa"]}), flush=True)
    if "parity" in parts:
        res["parity"] = parity(dev)
    res["card_after"] = card()
    print(json.dumps(res))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
