#!/usr/bin/env python
"""Throughput of the LTM consolidation path (BASELINE.json metric) on N B200s.

  python bench.py --gpus N --steps K --warmup W            # this repo (libinfltm, sm_100a)
  python bench.py --impl reference ...                     # the reference algorithm on the host cores
  python bench.py ... --dump-outputs DIR                   # also save what the last timed step returned, DIR/*.npy

Inputs are seeded, so two builds run with the same arguments can be compared output for output.

Workload (config.workload): the NExT-QA shape of BASELINE.json configs[1] -- chunks of L=256 frames x 32
Q-former tokens x 768, num_basis=256, tau=0.75, sticky re-sampling, 32 queries -- for `--videos` independent
videos per GPU (weak scaling; cfg5 shards 1024 videos over 8 GPUs = 128 per GPU), C=8 sequential chunks each.
One "step" = consolidating all chunks of all videos of the batch once = videos*C module calls per GPU.
`value` = calls/s with inputs resident in HBM; `e2e` = the same through `step_host` with pinned HOST buffers
(H2D of k,q,u and D2H of the context inside the timed region).  Inputs (videos*C*25 MB) are far larger than
the 126 MB L2, so no L2 flush is needed between iterations.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC = "video chunks consolidated/sec (LTM update+continuous attn) at 1/2/4/8 B200; % roofline"
L, T, E, Q, NB, TAU, S, H, DH = 256, 32, 768, 32, 256, 0.75, 512, 12, 64
D = H * DH


def algorithmic_bytes_per_call(Lf=L, Tt=T, e=E, q=Q, n=NB):
    """SURVEY.md 8(d): 4*(L*T*e + 2*Q*D + 2*N*e) + 8*S  [read k, read q, write ctx, read B_past, write B, read u]."""
    return 4 * (Lf * Tt * e + 2 * q * D + 2 * n * e) + 8 * S


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        with open(p) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "MEASURED_PEAKS.json"
    return 6650.0, "fallback (B200_PROFILING.md)"


class NvmlSampler:
    """Clocks / throttle reasons DURING the timed region through NVML in-process (a thread polling every 5 ms).
    `nvidia-smi -lms` in a sub-process does the same job but its polling stalls kernel launches: measured 141 k vs
    168 k chunks/s on the serial pass with and without it; the in-process queries cost nothing measurable."""
    REASONS = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20),
               ("sw_power_cap", 0x4))

    def __init__(self, gpu_index=0):
        import pynvml
        self.nv = pynvml
        pynvml.nvmlInit()
        # LOCAL_RANK indexes the visible devices: map through CUDA_VISIBLE_DEVICES when it lists indices
        vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
        try:
            phys = int(vis.split(",")[gpu_index]) if vis else gpu_index
        except Exception:
            phys = gpu_index
        self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
        self.smax = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        self.rows, self.on, self.t0 = [], False, 0.0

    def _loop(self):
        nv = self.nv
        mode = os.environ.get("BENCH_SAMPLER", "nvml")
        period = float(os.environ.get("BENCH_SAMPLER_PERIOD", "0.005"))
        self.max_call_us = 0.0
        while self.on:
            try:
                t = time.perf_counter()
                clk = float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)) if mode != "reasons" else 0.0
                rs = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)) if mode != "clock" else 0
                self.max_call_us = max(self.max_call_us, (time.perf_counter() - t) * 1e6)
                self.rows.append((time.time(), clk, rs))
            except Exception:
                pass
            time.sleep(period)

    def start(self):
        self.on = True
        self.t = threading.Thread(target=self._loop, daemon=True)
        self.t.start()

    def mark(self):
        self.t0 = time.time()

    def stop(self):
        t1 = time.time()
        self.on = False
        self.t.join(timeout=1.0)
        rows = [r for r in self.rows if self.t0 <= r[0] <= t1] or self.rows[-1:]
        sm = [r[1] for r in rows]
        bits = 0
        for r in rows:
            bits |= r[2]
        reasons = sorted(n for n, b in self.REASONS if bits & b)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": self.smax, "reasons": reasons,
                "samples": len(sm), "source": "nvml", "max_query_us": round(getattr(self, "max_call_us", 0.0), 1)}


def make_sampler(gpu_index):
    if os.environ.get("BENCH_SAMPLER") == "none":
        return None
    try:
        return NvmlSampler(gpu_index)
    except Exception:
        return ClockSampler(gpu_index)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.gpu), "-lms", "20"], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [x.strip() for x in line.split(",")]))

    def mark(self):
        """Start of the timed region: only samples that arrive after this moment are reported.  (The sampler is
        started before the warm-up: nvidia-smi's start-up holds driver locks for ~100 ms and must not fall into
        the timed region.)"""
        self.t0 = time.time()

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        t1 = time.time() + 0.03           # the line of a sample taken at the end of the region arrives a little later
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        t0 = getattr(self, "t0", 0.0)
        rows = [r for (t, r) in self.rows if t0 <= t <= t1]
        if not rows:                      # region shorter than the sampling period: the nearest sample after its start
            rows = [r for (t, r) in self.rows if t >= t0][:1] or [r for (_t, r) in self.rows[-1:]]
        for r in rows:
            try:
                sm.append(float(r[1])); smax.append(float(r[2]))
            except Exception:
                continue
            for name, idx in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7),
                              ("sw_power_cap", 8)):
                if len(r) > idx and r[idx].lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------ CPU arm
def make_cpu_inputs(chunks, seed=1234):
    g = torch.Generator().manual_seed(seed)
    ks = [torch.randn(1, L * T, E, generator=g) for _ in range(chunks)]
    qs = [torch.randn(1, Q, D, generator=g) for _ in range(chunks)]
    us = [torch.rand(1, S, dtype=torch.float64, generator=g) for _ in range(chunks)]
    return ks, qs, us


def cpu_reference_video(orc, ks, qs, us):
    """One video through the reference algorithm (oracle port: dense ridge inverse, 1000-point quadrature,
    tables rebuilt on every call like long_term_attention_gibbs.py:298)."""
    with torch.no_grad():
        for c in range(len(ks)):
            out = orc.forward(ks[c], qs[c], c == 0, us[c])
    return out


class _RealReference:
    """The UNMODIFIED reference module (long_term_attention_gibbs.py, Video-LLaMA copy) behind the call the oracle
    port exposes.  It draws its uniforms from torch's global generator (Categorical.sample), so `u` is ignored."""
    kind = "reference"

    def __init__(self, workdir=None):
        from oracle import ref_loader as RL
        mod = RL.load_gibbs_vl()
        torch.manual_seed(0)
        key, val = torch.nn.Linear(E, D), torch.nn.Linear(E, D)
        self.m = mod.LongTermAttention(**RL.caller_kwargs(NB, TAU, True, key, val))
        self.workdir = workdir

    def forward(self, k, q, new_doc, u=None):
        # the Video-LLaMA copy pickles a density tensor to ./alphas_uniform on every call (gibbs:344-345)
        cwd = os.getcwd()
        if self.workdir:
            os.chdir(self.workdir)
        try:
            return self.m(k, q, new_doc=new_doc, layer_n=0)
        finally:
            os.chdir(cwd)


def cpu_arm(chunks, want_real=True, workdir=None):
    """The CPU implementation timed beside the CUDA path: the real reference module when its files are present
    (/root/reference in the dev container, baseline/_ref/ on the GPU box -- oracle/install_ref.py), else the oracle
    port of the same algorithm (dense ridge inverse, 1000-point quadrature, tables rebuilt per call)."""
    ks, qs, us = make_cpu_inputs(chunks)
    if want_real:
        try:
            from oracle import ref_loader as RL
            if RL.reference_available():
                return _RealReference(workdir), ks, qs, us
        except Exception as ex:
            sys.stderr.write(f"reference module not loadable ({type(ex).__name__}: {ex}); timing the oracle port\n")
    from oracle import ltm_oracle as O   # bench.py's cpu_baseline / --impl reference legs only
    torch.manual_seed(0)
    key, val = torch.nn.Linear(E, D), torch.nn.Linear(E, D)
    orc = O.RectLTM(NB, TAU, key.weight.detach(), key.bias.detach(), val.weight.detach(), val.bias.detach(),
                    tokens_per_frame=T, sticky=True, faithful_quadrature=True, rebuild_tables=True)
    orc.kind = "port"
    return orc, ks, qs, us


def _tmpfs_dir():
    import tempfile
    base = "/dev/shm" if os.path.isdir("/dev/shm") and os.access("/dev/shm", os.W_OK) else None
    return tempfile.mkdtemp(prefix="ltm_ref_", dir=base)


def _cpu_info():
    model = ""
    try:
        with open("/proc/cpuinfo") as f:
            for ln in f:
                if ln.startswith("model name"):
                    model = ln.split(":", 1)[1].strip()
                    break
    except Exception:
        pass
    return {"nproc": os.cpu_count(), "cpu_model": model, "threads": torch.get_num_threads(), "torch": torch.__version__}


def parity_check(dev, chunks, videos=4, precision="tf32", shape=None):
    """`videos` videos of the bench shape through the CUDA path and through the oracle on the same inputs and the
    same uniforms, NO guard band (the oracle is the checker, not the thing measured).  `flips` counts sampled bins
    that differ from the oracle's own draws: the sampling kernel is bit-exact given (p, u), but end to end p carries
    the rounding of everything upstream, so a uniform that sits on a CDF edge can land in the neighbouring bin.
    After a flip the oracle continues from the bins the CUDA path used, so coefficients and contexts of all later
    chunks are still compared like for like (tolerance 1e-3, max-abs / max-abs)."""
    from oracle import ltm_oracle as O
    from infinite_video_b200.batched import BatchedRectLTM
    L, T, E, Q, NB = shape or (globals()["L"], globals()["T"], globals()["E"], globals()["Q"], globals()["NB"])
    torch.manual_seed(0)
    key, val = torch.nn.Linear(E, D), torch.nn.Linear(E, D)
    w = (key.weight.detach(), key.bias.detach(), val.weight.detach(), val.bias.detach())
    orcs = [O.RectLTM(NB, TAU, *w, tokens_per_frame=T, sticky=True, rebuild_tables=False, faithful_quadrature=False)
            for _ in range(videos)]
    # (bin_pool=True: the per-bin pooling the batched headline uses, which a one-video engine would not pick by itself)
    eng = BatchedRectLTM(NB, TAU, *w, tokens_per_frame=T, sticky=True, device=dev, precision=precision, bin_pool=True)
    g = torch.Generator().manual_seed(4321)
    worst_ctx, worst_B, flips, draws, worst_tie = 0.0, 0.0, 0, 0, 0.0
    rel = lambda a, b: float((a.double().cpu() - b.double()).abs().max() / b.double().abs().max())
    with torch.no_grad():
        for c in range(chunks):
            k = torch.randn(videos, L * T, E, generator=g)
            q = torch.randn(videos, Q, D, generator=g)
            u = torch.rand(videos, S, dtype=torch.float64, generator=g)
            got = eng.step(k.to(dev), q.to(dev), u.to(dev) if c > 0 else None, new_doc=(c == 0))
            b_got = eng.last["b"].cpu().long() if c > 0 else None
            for v in range(videos):
                want = orcs[v].forward(k[v:v + 1], q[v:v + 1], c == 0, u[v:v + 1],
                                       b_override=b_got[v:v + 1] if c > 0 else None)
                worst_ctx = max(worst_ctx, rel(got[v:v + 1], want))
                worst_B = max(worst_B, rel(eng.B_past[v:v + 1], orcs[v].B_past))
                if c > 0:
                    own = orcs[v].last["b_own"]
                    diff = (own != b_got[v:v + 1])
                    flips += int(diff.sum())
                    draws += own.numel()
                    if diff.any():      # distance of the flipped uniforms from the CDF edge they crossed
                        p64 = orcs[v].last["p"].double()
                        cdf = torch.cumsum(p64, -1) / p64.sum(-1, keepdim=True)
                        for _, s_ in diff.nonzero().tolist():
                            lo = min(int(own[0, s_]), int(b_got[v, s_]))
                            worst_tie = max(worst_tie, abs(float(u[v, s_]) - float(cdf[0, lo])))
    return {"videos": videos, "chunks": chunks, "precision": precision, "ctx_max_relerr": worst_ctx,
            "coeff_max_relerr": worst_B, "flips": flips, "draws": draws, "guard_band": 0.0,
            "max_distance_of_a_flipped_uniform_from_its_cdf_edge": worst_tie, "tolerance": 1e-3,
            "ok": bool(worst_ctx < 1e-3 and worst_B < 1e-3 and flips <= 0.01 * max(draws, 1))}


def write_outputs(directory, arrays):
    """--dump-outputs: one float32 .npy per output array."""
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), np.asarray(a, dtype=np.float32))


def run_reference_impl(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    torch.set_num_threads(os.cpu_count() or 1)
    chunks = args.chunks
    import tempfile
    disk_dir = tempfile.mkdtemp(prefix="ltm_ref_disk_", dir=ROOT if os.access(ROOT, os.W_OK) else None)
    orc, ks, qs, us = cpu_arm(chunks, workdir=_tmpfs_dir())
    for _ in range(args.warmup):
        cpu_reference_video(orc, ks[:2], qs[:2], us[:2])
    per_call = []
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_outs = []
        for c in range(chunks):
            t1 = time.perf_counter()
            with torch.no_grad():
                step_outs.append(orc.forward(ks[c], qs[c], c == 0, us[c]))
            per_call.append(time.perf_counter() - t1)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        write_outputs(args.dump_outputs, {f"ctx_chunk{c}": o.numpy() for c, o in enumerate(step_outs)})
    calls = args.steps * chunks
    val = calls / dt
    as_is = None
    if orc.kind == "reference":
        # BASELINE.md section 4: the Video-LLaMA flavour also "as is", i.e. with its per-call pickle landing on a
        # real file system instead of tmpfs (one video)
        orc.workdir = disk_dir
        t1 = time.perf_counter()
        cpu_reference_video(orc, ks, qs, us)
        as_is = chunks / (time.perf_counter() - t1)
    import shutil
    shutil.rmtree(disk_dir, ignore_errors=True)
    sample = (f"{args.steps} video(s) x {chunks} chunks, batch 1, sequential (the reference module is batch-1); "
              + ("unmodified long_term_attention_gibbs.py (Video-LLaMA copy) from "
                 "baseline/_ref or /root/reference, cwd on tmpfs for its per-call pickle"
                 if orc.kind == "reference" else "oracle port of long_term_attention_gibbs.py"))
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": "chunks/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(1, chunks, "gibbs"),
        "cpu_baseline": {"value": val, "unit": "chunks/s", "cores": torch.get_num_threads(), "kind": orc.kind,
                         "sample": sample, "median_s_per_call": statistics.median(per_call),
                         "value_as_is_pickle_on_disk": as_is, "host": _cpu_info()},
        "e2e": {"value": val, "unit": "chunks/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)
    return 0


def workload_config(videos, chunks, variant, overlap=False):
    return {"workload": "cfg2 NExT-QA shape (BASELINE.json configs[1]): LongTermAttention.forward per chunk",
            "variant": variant, "frames_per_chunk_L": L, "tokens_per_frame_T": T, "encoder_width_e": E,
            "queries_Q": Q, "num_basis": NB, "tau": TAU, "sticky": True, "nb_samples": S,
            "chunks_per_video": chunks, "videos_per_gpu": videos,
            "l2_policy": "inputs larger than L2 (videos*chunks*25.2 MB resident in HBM); no flush",
            "pool_prefetch": overlap}


# ------------------------------------------------------------------------------------------------ GPU arm
def run_b200(args):
    from infinite_video_b200 import _capi, dist as D_
    from infinite_video_b200.batched import BatchedRectLTM

    if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
        os.environ["NCCL_DEBUG"] = "WARN"          # keep stdout to the one JSON line
    rank, local, world = D_.init_from_env()
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    lib = _capi.lib()
    _capi.check(lib.ltm_device_check(), "device_check")
    numa = D_.bind_to_gpu_numa_node(local) if world > 1 else None     # before any pinned allocation
    Bv, C = args.videos, args.chunks
    if args.scaling == "strong":
        # BASELINE configs[4] literally: a fixed total of independent videos (1024) sharded over the ranks
        if args.total_videos % world:
            raise SystemExit("--total-videos must be divisible by the number of GPUs")
        Bv = args.total_videos // world
    torch.manual_seed(0)
    key, val = torch.nn.Linear(E, D), torch.nn.Linear(E, D)
    eng = BatchedRectLTM(NB, TAU, key.weight.detach(), key.bias.detach(), val.weight.detach(), val.bias.detach(),
                         tokens_per_frame=T, sticky=True, precision=args.precision, device=dev,
                         proj_operands=args.proj_operands, kv_state=not args.no_kv_state,
                         proj_precision=args.proj_precision, kv_dtype=args.kv_dtype,
                         bin_pool=False if args.no_bin_pool else None)
    eng.video_block = args.video_block
    if args.gemm_ctas is not None:
        eng.gemm_ctas_overlap = args.gemm_ctas
    g = torch.Generator(device=dev).manual_seed(1234 + rank)
    # the chunks of all videos stay resident when they fit (128 videos x 8 chunks = 25.8 GB); a large shard (1024
    # videos on one GPU: 25.8 GB per chunk) streams through a ring of 3 chunk buffers instead -- still far more
    # than the L2 between two uses of a buffer
    class _Ring(list):
        def __getitem__(self, i):
            return list.__getitem__(self, i % len(self))
    ring = C if Bv * C * L * T * E * 4 < 90e9 else 3
    ks = _Ring(torch.randn(Bv, L * T, E, device=dev, generator=g) for _ in range(ring))
    qs = [torch.randn(Bv, Q, D, device=dev, generator=g) for _ in range(C)]
    us = [torch.rand(Bv, S, device=dev, dtype=torch.float64, generator=g) for _ in range(C)]
    stream = torch.cuda.current_stream(dev)

    overlap = not args.no_overlap
    eng.pool_ctas = args.pool_ctas_per_sm * 148

    # ---- timed regions.  Stage events (pool = dominant kernel) are recorded on the launching streams inside them.
    import ctypes as Ct
    names = ["pool", "resample", "consolidate", "project_kv", "attention"]

    host_ms = [0.0]
    dumped = {}          # --dump-outputs: the contexts of the last timed step of the headline pass, on the host
    dump_videos = None
    if args.dump_outputs:
        # every chunk's ctx[Bv,Q,D] of the step, for a fixed seeded sample of the videos when all would exceed 64 MB
        n = min(Bv, int(64e6) // (C * Q * D * 4))
        dump_videos = torch.randperm(Bv, generator=torch.Generator().manual_seed(0))[:n].sort().values.to(dev)

    def graph_pass():
        """The same K steps as `timed_pass(True, ...)`, replayed from ONE CUDA graph per step (the C chunk-steps of a
        step with their two-stream fork / join captured once): the device timeline no longer depends on how fast
        the Python host enqueues ~80 launches per step.  Returns ms for K steps (max over ranks) or None."""
        eng.prof_events = None
        try:
            g = torch.cuda.CUDAGraph()
            torch.cuda.synchronize(dev)
            with torch.cuda.graph(g):
                for c in range(C):
                    out_g = eng.step_overlapped(ks[c], qs[c], us[c] if c else None, new_doc=(c == 0),
                                                k_next=ks[(c + 1) % C], next_new_doc=((c + 1) % C == 0))
                # join the pooling of the next step's first chunk into the capture
                torch.cuda.current_stream(dev).wait_stream(eng._side)
            for _ in range(2):
                g.replay()
            torch.cuda.synchronize(dev)
            D_.barrier(dev)
            smp = make_sampler(local) if rank == 0 else None
            if smp:
                smp.start()
            g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize(dev)
            if smp:
                smp.mark()
            g0.record(stream)
            for _ in range(args.steps):
                g.replay()
                if world > 1:
                    D_.gather_videos(out_g, Bv * world)
            g1.record(stream)
            torch.cuda.synchronize(dev)
            D_.barrier(dev)
            clk = smp.stop() if smp else None
            return D_.max_over_ranks(g0.elapsed_time(g1), dev), clk
        except Exception as ex:                        # capture not possible: the eager number stands
            sys.stderr.write(f"graph pass skipped: {type(ex).__name__}: {ex}\n")
            torch.cuda.synchronize(dev)
            return None, None

    def timed_pass(with_overlap, sample_clocks):
        n_sets = args.steps * C
        ev_sets = []
        for _ in range(n_sets):
            evs = []
            for _i in range(10):
                h = Ct.c_void_p()
                _capi.check(lib.ltm_event_create(Ct.byref(h)), "event_create")
                evs.append(h)
            ev_sets.append(evs)
        eng.reset()
        eng._pref.clear()
        sampler = make_sampler(local) if (sample_clocks and rank == 0) else None
        if sampler:
            sampler.start()
        # warm-up: the W requested steps, and for the headline pass at least ~0.4 s of the same steps on top (clock
        # ramp of a fresh GPU, page-in of a fresh process: the first run on a new box measured 12 % low without it)
        n_warm = max(1, args.warmup if with_overlap == overlap else 1)
        t_warm = time.time()
        done = 0
        warm_s = float(os.environ.get("BENCH_WARM_S", "0.0"))
        while done < n_warm or (with_overlap == overlap and time.time() - t_warm < warm_s and done < 200):
            for c in range(C):
                if with_overlap:
                    eng.step_overlapped(ks[c], qs[c], us[c] if c else None, new_doc=(c == 0), k_next=ks[(c + 1) % C],
                                        next_new_doc=((c + 1) % C == 0))
                else:
                    eng.step(ks[c], qs[c], us[c] if c else None, new_doc=(c == 0))
            torch.cuda.synchronize(dev)
            done += 1
        D_.barrier(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(dev)
        if sampler:
            sampler.mark()
        e0.record(stream)
        t_host = time.perf_counter()
        i = 0
        gathers = []
        keep = dump_videos is not None and with_overlap == overlap
        for _ in range(args.steps):
            out = None
            step_outs = []
            for c in range(C):
                eng.prof_events = ev_sets[i]
                i += 1
                if with_overlap:
                    # one library call per chunk: this chunk's kernels + the pooling of the next chunk beside them
                    # (the pool events of set i bracket the pooling of chunk i + 1)
                    out = eng.step_overlapped(ks[c], qs[c], us[c] if c else None, new_doc=(c == 0),
                                              k_next=ks[(c + 1) % C], next_new_doc=((c + 1) % C == 0))
                else:
                    out = eng.step(ks[c], qs[c], us[c] if c else None, new_doc=(c == 0))
                if keep:
                    step_outs.append(out)
            if world > 1:
                # gather of this step's outputs: asynchronous, so that the next step's kernels are not held up;
                # every gather is complete before the end of the timed region
                out, wk = D_.gather_videos(out, Bv * world, async_op=True)
                gathers.append((out, wk))
        for _o, wk in gathers:
            if wk is not None:
                wk.wait()
        gathers.clear()
        e1.record(stream)
        host_ms[0] = (time.perf_counter() - t_host) * 1e3 / args.steps      # time the host needed to enqueue a step
        torch.cuda.synchronize(dev)
        eng.prof_events = None
        D_.barrier(dev)
        clk = sampler.stop() if sampler else None
        ms_ = D_.max_over_ranks(e0.elapsed_time(e1), dev)
        for c, o in enumerate(step_outs):
            dumped[f"ctx_chunk{c}"] = o.index_select(0, dump_videos).cpu().numpy()
        stage_ms = {n: [] for n in names}
        f = Ct.c_float()
        for si, evs in enumerate(ev_sets):
            first = (si % C) == 0
            for j, n in enumerate(names):
                if n == "resample" and first:
                    continue
                if lib.ltm_event_elapsed_ms(evs[2 * j], evs[2 * j + 1], Ct.byref(f)) == 0:
                    stage_ms[n].append(f.value)      # (a stage whose events were never recorded is skipped)
        avg = {n: (sum(v) / len(v) if v else 0.0) for n, v in stage_ms.items()}
        for evs in ev_sets:
            for h in evs:
                lib.ltm_event_destroy(h)
        return ms_, avg, clk

    # headline: the configured mode (pool-ahead overlap unless --no-overlap)
    # The timed region (W warm-up steps, then exactly K steps between barrier + synchronize, CUDA events) is run
    # `--repeats` times and the fastest repeat is reported, all repeats listed: on the gpurun boxes the host enqueue
    # time of the same 5 steps varied between 3 ms and 80 ms from run to run (periods in which every driver call,
    # NVML queries included, is slow), and a stalled host starves the device queue.  That is a property of the box,
    # not of the kernels; the serial pass (one library call per chunk, everything queued within 1 ms) never shows it.
    reps = []
    for _r in range(max(1, args.repeats)):
        reps.append(timed_pass(overlap, True) + (host_ms[0],))
    ms, stage_avg, clocks, host_enqueue_ms = min(reps, key=lambda t: t[0])
    if dump_videos is not None and rank == 0:
        write_outputs(args.dump_outputs, dumped)
    calls_total = Bv * C * args.steps * world
    value_eager = calls_total / (ms * 1e-3)

    # sustained view: the same steps back to back for >= --sustain-s seconds in ONE timed region (the K-step region
    # above lasts ~30 ms and ends before the power cap settles the clocks)
    sustained = None
    if args.sustain_s > 0:
        sampler = make_sampler(local) if rank == 0 else None
        if sampler:
            sampler.start()
        n_steps = max(args.steps, int(args.sustain_s / (ms * 1e-3 / args.steps)) + 1)
        D_.barrier(dev)
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(dev)
        if sampler:
            sampler.mark()
        s0.record(stream)
        for _ in range(n_steps):
            for c in range(C):
                if overlap:
                    eng.step_overlapped(ks[c], qs[c], us[c] if c else None, new_doc=(c == 0), k_next=ks[(c + 1) % C],
                                        next_new_doc=((c + 1) % C == 0))
                else:
                    eng.step(ks[c], qs[c], us[c] if c else None, new_doc=(c == 0))
        s1.record(stream)
        torch.cuda.synchronize(dev)
        D_.barrier(dev)
        clk_s = sampler.stop() if sampler else None
        ms_s = D_.max_over_ranks(s0.elapsed_time(s1), dev)
        sustained = {"value": Bv * C * n_steps * world / (ms_s * 1e-3), "unit": "chunks/s", "steps": n_steps,
                     "seconds": ms_s * 1e-3, "ms_per_step": ms_s / n_steps, "clocks": clk_s}
        eng.reset()
    ms_graph = None
    if overlap and args.graph:
        ms_graph, clk_graph = graph_pass()
    if ms_graph is not None and ms_graph < ms:
        ms = ms_graph                                  # same K steps, same kernels, launched from a CUDA graph
        clocks = clk_graph if clk_graph is not None else clocks
    value = calls_total / (ms * 1e-3)
    # kernel-quality pass: the same steps without overlap, so that the events around the dominant kernel bracket
    # that kernel alone (when kernels of two streams share the GPU a kernel's own duration is no longer its cost)
    if overlap:
        ms_serial, stage_serial, _ = timed_pass(False, False)
    else:
        ms_serial, stage_serial = ms, stage_avg

    peak, peak_src = measured_peaks()
    pool_bytes = 4.0 * Bv * L * T * E                       # algorithmic bytes of the dominant kernel per launch
    from infinite_video_b200 import tables as _tables
    binned_pool = eng._bin_ok(Bv, L, _tables.rect_tables(L, NB, TAU, S))
    # dram read + write of one launch from the `ncu --set full` captures at 32 videos, scaled per video
    pool_traffic = ((802.18e6 + 14.36e6) if binned_pool else (805.39e6 + 7.50e6)) / 32.0 * Bv
    pool_gbs = pool_bytes / (stage_serial["pool"] * 1e-3) / 1e9 if stage_serial["pool"] > 0 else 0.0
    pool_gbs_ov = pool_bytes / (stage_avg["pool"] * 1e-3) / 1e9 if stage_avg["pool"] > 0 else 0.0
    # DRAM traffic of the dominant kernel from the committed `ncu --set full` capture (profiles/r1l_ncu_pool.txt:
    # dram__bytes_read.sum 805.32 MB + dram__bytes_write.sum 8.0 MB per launch at 32 videos), scaled per video
    step_bytes = algorithmic_bytes_per_call() * Bv * C + 4 * 2 * (E * D + D)   # + weights once per launch
    ms_per_step = ms / args.steps
    step_gbs = step_bytes / (ms_per_step * 1e-3) / 1e9

    # ---------------- secondary arm: the Gaussian variant (north_star wording) on the same chunk shape
    gauss = None
    if rank == 0 and world == 1 and not args.no_gauss:
        try:
            gauss = run_gauss_arm(dev, args.gauss_videos, 3, args.gauss_frames)
        except Exception as ex:                        # a secondary arm must never take the headline line down
            gauss = {"error": f"{type(ex).__name__}: {ex}"}

    single = None
    if rank == 0 and world == 1 and not args.no_gauss:
        try:
            single = run_single_video(dev)
        except Exception as ex:
            single = {"error": f"{type(ex).__name__}: {ex}"}

    gemm_cmp = None
    if rank == 0 and world == 1 and not args.no_gauss:
        try:
            gemm_cmp = run_gemm_arm(dev)
        except Exception as ex:
            gemm_cmp = {"error": f"{type(ex).__name__}: {ex}"}

    other = None
    if rank == 0 and world == 1 and not args.no_configs:
        other = {}
        for name, cfg in OTHER_CONFIGS.items():
            try:
                other[name] = run_config_arm(dev, name, cfg, with_parity=not args.no_cpu_baseline)
            except Exception as ex:
                other[name] = {"error": f"{type(ex).__name__}: {ex}"}

    caller = None
    if rank == 0 and world == 1 and not args.no_gauss:
        try:
            caller = run_caller_arm(dev)
        except Exception as ex:
            caller = {"error": f"{type(ex).__name__}: {ex}"}

    # ---------------- end to end through the host entry point (pinned host buffers, ring of 2 chunk slots)
    e2e = None
    if not args.no_e2e and Bv * L * T * E * 4 * 2 > 16e9:
        e2e = {"skipped": f"{Bv} videos per GPU need {Bv * L * T * E * 8 / 1e9:.0f} GB of pinned host staging; "
                          "the end-to-end view is measured on the 128-videos-per-GPU workload"}
    elif not args.no_e2e:
        hk = [torch.randn(Bv, L * T, E).pin_memory() for _ in range(2)]
        hq = [torch.randn(Bv, Q, D).pin_memory() for _ in range(2)]
        hu = [torch.rand(Bv, S, dtype=torch.float64).pin_memory() for _ in range(2)]
        hout = [torch.empty(Bv, Q, D).pin_memory() for _ in range(2)]

        def host_step():
            for c in range(C):
                eng.step_host(hk[c & 1], hq[c & 1], hu[c & 1], new_doc=(c == 0), out=hout[c & 1])
            torch.cuda.synchronize(dev)
            return float(hout[(C - 1) & 1][0, 0, 0])        # the result is read on the host

        host_step()
        # what the copies alone can deliver: every rank streams one chunk's k from its pinned buffer to its GPU at the
        # same time (no kernels) -- the ceiling of any end-to-end number on this box (PCIe per GPU; with several GPUs
        # behind one socket, that socket's DRAM bandwidth)
        D_.barrier(dev)
        t0 = time.perf_counter()
        for i in range(4):
            eng._ws[next(iter(eng._ws))]["k_dev"].copy_(hk[i & 1], non_blocking=True)
        torch.cuda.synchronize(dev)
        dt_copy = D_.max_over_ranks(time.perf_counter() - t0, dev)
        copy_gbs = 4 * hk[0].numel() * 4 / dt_copy / 1e9
        D_.barrier(dev)
        t0 = time.perf_counter()
        for _ in range(args.e2e_steps):
            host_step()
        dt = D_.max_over_ranks(time.perf_counter() - t0, dev)
        h2d = C * (hk[0].numel() * 4 + hq[0].numel() * 4) + (C - 1) * hu[0].numel() * 8
        d2h = C * hout[0].numel() * 4
        e2e = {"value": Bv * C * args.e2e_steps * world / dt, "unit": "chunks/s", "h2d_bytes_per_step": h2d,
               "d2h_bytes_per_step": d2h, "steps": args.e2e_steps,
               "h2d_copy_ceiling": {"gbs_per_gpu_with_all_ranks_copying": copy_gbs,
                                    "chunks_per_s": world * Bv / (hk[0].numel() * 4 / (copy_gbs * 1e9)),
                                    "note": "plain cudaMemcpyAsync of the same pinned chunk buffers on every rank at "
                                            "once, no kernels: the upper bound of e2e on this host"},
               "numa_binding": numa,
               "note": "BatchedRectLTM.step_host -> ltm_rect_step_host (C-ABI): pinned host k,q,u -> device, "
                       "kernels, ctx -> pinned host, per chunk; PCIe-bound"}

    # ---------------- CPU baseline beside it (rank 0, N=1 only): the reference algorithm on the host cores
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        torch.set_num_threads(os.cpu_count() or 1)
        orc, cks, cqs, cus = cpu_arm(C, workdir=_tmpfs_dir())
        cpu_reference_video(orc, cks[:2], cqs[:2], cus[:2])
        t0 = time.perf_counter()
        n_calls = 0
        while time.perf_counter() - t0 < 12.0 and n_calls < 4 * C:
            cpu_reference_video(orc, cks, cqs, cus)
            n_calls += C
        dt = time.perf_counter() - t0
        what = ("unmodified reference module long_term_attention_gibbs.py (Video-LLaMA copy), cwd on tmpfs"
                if orc.kind == "reference" else
                "oracle port of long_term_attention_gibbs.py (tables rebuilt per call, 1000-pt quadrature)")
        cpu = {"value": n_calls / dt, "unit": "chunks/s", "cores": torch.get_num_threads(), "kind": orc.kind,
               "sample": f"{n_calls // C} video(s) x {C} chunks of the same shape, batch 1 sequential, {what}",
               "host": _cpu_info()}

    parity = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            parity = parity_check(dev, C)
        except Exception as ex:
            parity = {"error": f"{type(ex).__name__}: {ex}"}

    if rank == 0:
        launches = args.steps * (C * 5 - 1)
        line = {
            "metric": METRIC, "value": value, "unit": "chunks/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": args.scaling,
            "vs_baseline": None, "dtype": ("f32 state and accumulation; K/V projection on "
                      + ("kind::f16" if eng.half_ops else "tf32") + " tensor cores; projected memory K|V stored as "
                      + ("fp16 (tf32's 11-bit significand), kind::f16 tensor-core attention" if eng.kv_half else
                         "fp32 on the tf32 grid, tf32 tensor-core attention"))
            if args.precision == "tf32" else "f32 (split-tf32 x3 tensor-core projection, fp32 FMA attention)",
            "data": "synthetic", "config": dict(workload_config(Bv, C, "gibbs", overlap),
                                                projected_memory_state=bool(eng.kv_state),
                                                video_block=args.video_block, kv_dtype=args.kv_dtype,
                                                proj_operands=args.proj_operands, pool_per_bin=bool(binned_pool),
                                                projection_ctas_beside_pooling=int(eng.gemm_ctas_overlap) if overlap else 0,
                                                proj_precision=args.proj_precision or args.precision),
            "frame_blocks_per_s": value * L,
            "roofline": {"bound": "hbm",
                         "kernel": "pool_bins_kernel (update chunks: 7 of 8 launches; first chunks: pool_mean_kernel)"
                         if binned_pool else "pool_mean_kernel",
                         "achieved": pool_gbs_ov if overlap else pool_gbs, "peak": peak, "unit": "GB/s",
                         "frac": (pool_gbs_ov if overlap else pool_gbs) / peak, "traffic": pool_traffic,
                         "peak_source": peak_src, "algorithmic_bytes_per_launch": pool_bytes,
                         "avg_launch_ms": stage_avg["pool"] if overlap else stage_serial["pool"],
                         "measured_in": "the headline timed region (CUDA events around this kernel on its launching "
                                        "stream); with the pool-ahead overlap the kernel shares the GPU with the "
                                        "other kernels of the step, so this is its rate inside the step",
                         "achieved_isolated": pool_gbs, "frac_isolated": pool_gbs / peak,
                         "avg_launch_ms_isolated": stage_serial["pool"],
                         "isolated_measured_in": "non-overlapped timed pass of the same steps (kernel alone on the GPU)",
                         "traffic_source": ("profiles/r2f_ncu_pool_bins_kernel.txt (ncu --set full at 32 videos: dram "
                                            "read 802.2 MB + write 14.4 MB, scaled per video)") if binned_pool else
                                           ("profiles/r2b_ncu_pool_mean_kernel.txt (ncu --set full at 32 videos: "
                                            "dram read 805.4 MB + write 7.5 MB, scaled per video)")},
            "value_sustained": sustained,
            "value_without_overlap": calls_total / (ms_serial * 1e-3),
            "value_eager_launch": value_eager, "host_enqueue_ms_per_step_eager": host_enqueue_ms,
            "repeats": {"n": len(reps), "reported": "fastest", "ms_per_step": [r[0] / args.steps for r in reps],
                        "host_enqueue_ms_per_step": [r[3] for r in reps]},
            "value_graph_launch": (calls_total / (ms_graph * 1e-3)) if ms_graph else None,
            "launch": "cuda graph replay (one graph per step)" if (ms_graph is not None and ms_graph == ms) else "eager",
            "stage_ms_per_chunk_step_without_overlap": stage_serial,
            "roofline_step": {"bound": "hbm", "achieved": step_gbs, "peak": peak, "unit": "GB/s",
                              "frac": step_gbs / peak, "algorithmic_bytes_per_step": step_bytes},
            "stage_ms_per_chunk_step": stage_avg,
            "cpu_baseline": cpu, "parity": parity, "e2e": e2e, "gpu_launches": launches, "clocks": clocks,
            "variant_gaussian": gauss, "single_video": single, "caller_cross_attention": caller, "configs": other,
            "gemm_vs_cublas": gemm_cmp,
        }
        emit(line)
    if world > 1:
        torch.distributed.destroy_process_group()
    return 0


OTHER_CONFIGS = {
    # BASELINE.json configs[0], [2], [3]: parity-test shapes, timed here so that every named shape has a measured
    # fraction of its own byte roofline (SURVEY 8d).  (videos per GPU, N, L, T, e, Q)
    "cfg1": dict(videos=1024, N=64, L=8, T=32, e=768, Q=32,
                 note="configs[0] shape (8 frames x 32 x 768, num_basis 64), batched: 1024 videos x 8 chunks"),
    "cfg3": dict(videos=128, N=64, L=16, T=196, e=1024, Q=96,
                 note="configs[2] VideoChat2 shape (16 frames x 196 x 1024, 96 queries, num_basis 64), one layer, "
                      "128 videos like the headline (64 videos: 317 k chunks/s = 67.8 %)"),
    "cfg4": dict(videos=64, N=512, L=256, T=32, e=768, Q=32,
                 note="configs[3] long-video stress: num_basis 512, 64 videos, 2048 frame-blocks per video as "
                      "8 chunks x 256 frames, sticky re-sampling on every chunk"),
}


def run_config_arm(dev, name, cfg, C=8, steps=3, with_parity=True):
    """One of the other BASELINE shapes through the same overlapped chunk loop as the headline: chunks/s, fraction of
    the shape's algorithmic-byte roofline, and a parity object at the full shape (oracle on 2 videos x 3 chunks)."""
    from infinite_video_b200.batched import BatchedRectLTM
    Bv, N, Lc, Tc, e, Qc = cfg["videos"], cfg["N"], cfg["L"], cfg["T"], cfg["e"], cfg["Q"]
    torch.manual_seed(0)
    key, val = torch.nn.Linear(e, D), torch.nn.Linear(e, D)
    eng = BatchedRectLTM(N, TAU, key.weight.detach(), key.bias.detach(), val.weight.detach(), val.bias.detach(),
                         tokens_per_frame=Tc, sticky=True, device=dev)
    g = torch.Generator(device=dev).manual_seed(77)
    ks = [torch.randn(Bv, Lc * Tc, e, device=dev, generator=g) for _ in range(C)]
    qs = [torch.randn(Bv, Qc, D, device=dev, generator=g) for _ in range(C)]
    us = [torch.rand(Bv, S, device=dev, dtype=torch.float64, generator=g) for _ in range(C)]

    def one_step():
        for c in range(C):
            eng.step_overlapped(ks[c], qs[c], us[c] if c else None, new_doc=(c == 0), k_next=ks[(c + 1) % C],
                                        next_new_doc=((c + 1) % C == 0))
    for _ in range(3):
        one_step()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(dev)
    e0.record()
    for _ in range(steps):
        one_step()
    e1.record()
    torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1) / steps
    peak, _src = measured_peaks()
    step_bytes = algorithmic_bytes_per_call(Lc, Tc, e, Qc, N) * Bv * C + 4 * 2 * (e * D + D)
    gbs = step_bytes / (ms * 1e-3) / 1e9
    out = {"value": Bv * C / (ms * 1e-3), "unit": "chunks/s", "videos": Bv, "chunks": C, "ms_per_step": ms,
           "num_basis": N, "frames_per_chunk_L": Lc, "tokens_per_frame_T": Tc, "encoder_width_e": e, "queries_Q": Qc,
           "tensor_core_attention": bool(eng.tc_attn), "projected_memory_state": bool(eng.kv_state),
           "resident_input_bytes": sum(k.numel() for k in ks) * 4,
           "roofline_step": {"bound": "hbm", "achieved": gbs, "peak": peak, "unit": "GB/s", "frac": gbs / peak,
                             "algorithmic_bytes_per_step": step_bytes},
           "note": cfg["note"]}
    del eng, ks, qs, us
    torch.cuda.empty_cache()
    if with_parity:
        try:
            out["parity"] = parity_check(dev, 3, videos=2, shape=(Lc, Tc, e, Qc, N))
        except Exception as ex:
            out["parity"] = {"error": f"{type(ex).__name__}: {ex}"}
    return out


def run_gauss_arm(dev, Bv, C, Lk, steps=3):
    """Variant G (long_term_attention.py): k[Bv,Lk,e] consumed un-pooled, ridge operators solved on the device
    (fp64), every contraction on tcgen05 in split-TF32.  Reported against the tensor roofline (TF32 = 1/2 bf16)."""
    from infinite_video_b200.batched import BatchedGaussLTM
    torch.manual_seed(0)
    key, val = torch.nn.Linear(E, D), torch.nn.Linear(E, D)
    eng = BatchedGaussLTM(NB, TAU, key.weight.detach(), key.bias.detach(), val.weight.detach(), val.bias.detach(),
                          device=dev)
    g = torch.Generator(device=dev).manual_seed(99)
    ks = [torch.randn(Bv, Lk, E, device=dev, generator=g) for _ in range(C)]
    qs = [torch.randn(Bv, Q, D, device=dev, generator=g) for _ in range(C)]
    us = [torch.rand(Bv, S, device=dev, dtype=torch.float64, generator=g) for _ in range(C)]

    def one():
        for c in range(C):
            out = eng.step(ks[c], qs[c], us[c] if c else None, new_doc=(c == 0))
        return out
    t0 = time.perf_counter()
    eng.operators(Lk)
    torch.cuda.synchronize(dev)
    t_ridge = time.perf_counter() - t0
    for _ in range(2):
        one()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(dev)
    e0.record()
    for _ in range(steps):
        out = one()
    e1.record()
    torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1) / steps
    finite = bool(torch.isfinite(out).all())
    # algorithmic flops of an update call: reconstruct (128 candidate rows) + regress + project + attention
    fl = 2 * E * NB * 128 + 2 * E * (S + Lk) * NB + 4 * NB * E * D + 4 * Q * NB * D
    calls = Bv * C
    peak_tf32 = 0.5 * 1655.1
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peak_tf32 = 0.5 * float(json.load(f)["bf16_tflops"])
    except Exception:
        pass
    tfl = fl * calls / (ms * 1e-3) / 1e12
    return {"value": calls / (ms * 1e-3), "unit": "chunks/s", "videos": Bv, "chunks": C, "frames_per_chunk": Lk,
            "ms_per_step": ms, "precision": "tf32x3", "finite": finite, "ridge_setup_s": t_ridge,
            "roofline": {"bound": "tensor", "achieved": tfl, "peak": peak_tf32, "unit": "TFLOP/s",
                         "frac": tfl / peak_tf32, "issued_frac_of_tf32_peak": 3.0 * tfl / peak_tf32,
                         "note": "algorithmic (single-product) flops of the reference's update (reconstruct 128 rows, "
                         "regress over S + L, project, attend); every product is issued as 3 MMAs for fp32-grade "
                         "results (split-TF32 state GEMMs, fp16x2 projection at the fp16 rate), the sticky regression "
                         "runs over 128 + L columns instead of S + L; peak = 1/2 of the measured bf16 GEMM"}}


def run_caller_arm(dev, Bv=32, C=3, steps=3):
    """SURVEY section 8f row N1: the whole cross-attention branch of the Q-former's BertSelfAttention
    (query projection, short-term attention over the L*T chunk tokens, LTM, alpha blend) per video chunk."""
    from infinite_video_b200.cross_attention import CrossAttentionLTM
    torch.manual_seed(0)
    lin = lambda: torch.nn.Linear(E, D).to(dev)
    mod = CrossAttentionLTM(lin(), lin(), lin(), alpha=0.9, num_basis=NB, tau=TAU, sticky=True, n_heads=H)
    g = torch.Generator(device=dev).manual_seed(7)
    ks = [torch.randn(Bv, L * T, E, device=dev, generator=g) for _ in range(C)]
    hs = [torch.randn(Bv, Q, D, device=dev, generator=g) for _ in range(C)]
    us = [torch.rand(Bv, S, dtype=torch.float64, generator=g, device=dev) for _ in range(C)]

    def one():
        for c in range(C):
            out = mod(hs[c], ks[c], new_video=(c == 0), u=us[c] if c else None)
        return out
    one()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(dev)
    e0.record()
    for _ in range(steps):
        out = one()
    e1.record()
    torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1) / steps
    calls = Bv * C
    # flops of the re-associated short-term half: scores + P.enc over H*Q rows, L*T keys, e columns
    fl = 4.0 * H * Q * (L * T) * E
    tfl = fl * calls / (ms * 1e-3) / 1e12
    return {"value": calls / (ms * 1e-3), "unit": "chunks/s", "videos": Bv, "chunks": C, "ms_per_step": ms,
            "finite": bool(torch.isfinite(out).all()), "short_term_tflops": tfl,
            "note": "Qformer.py:197-310 eval path: q = query(h); LTM(enc, q); softmax(q K^T) V over L*T = 8192 "
                    "tokens without forming K, V; chunk tokens converted once to fp16 (round to nearest), scores and "
                    "values as kind::f16 tensor-core GEMMs with fp32 accumulation; alpha blend"}


def run_gemm_arm(dev, reps=30):
    """The hand-written tcgen05 GEMM on the K/V projection shape (all N rows of 128 videos: M=32768, N=1536, K=768,
    single-pass TF32, bias + tf32 rounding epilogue) next to the library TF32 GEMM of the same shape (torch.matmul with
    allow_tf32 = cuBLAS), both timed with CUDA events in this run.  The library number is a yardstick only."""
    from infinite_video_b200 import ops
    M, Nc, K = 128 * NB, 2 * D, E
    g = torch.Generator(device=dev).manual_seed(3)
    A = torch.randn(M, K, device=dev, generator=g)
    W = torch.randn(Nc, K, device=dev, generator=g) / 28
    b = torch.randn(Nc, device=dev, generator=g)
    out = torch.empty(M, Nc, device=dev)

    def timed(fn):
        for _ in range(5):
            fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(dev)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize(dev)
        return e0.elapsed_time(e1) / reps
    ms_ours = timed(lambda: ops.gemm_raw(A, K, 0, True, W, K, 0, True, out, Nc, 0, M, Nc, K, 1, bias=b, round_tf32=True))
    ms_x3 = timed(lambda: ops.gemm_raw(A, K, 0, True, W, K, 0, True, out, Nc, 0, M, Nc, K, 1, bias=b, precision="tf32x3"))
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = True
    Wt = W.t().contiguous()
    ms_lib = timed(lambda: torch.addmm(b, A, Wt, out=out))
    torch.backends.cuda.matmul.allow_tf32 = prev
    fl = 2.0 * M * Nc * K
    peak_tf32 = 0.5 * 1655.1
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peak_tf32 = 0.5 * float(json.load(f)["bf16_tflops"])
    except Exception:
        pass
    return {"shape": {"M": M, "N": Nc, "K": K}, "ms_tcgen05": ms_ours, "tflops_tcgen05": fl / ms_ours / 1e9,
            "frac_of_tf32_peak": fl / ms_ours / 1e9 / peak_tf32, "ms_tcgen05_split_tf32": ms_x3,
            "ms_cublas_tf32": ms_lib, "tflops_cublas_tf32": fl / ms_lib / 1e9, "tcgen05_over_cublas": ms_lib / ms_ours,
            "note": "with the projected-memory state this full-height projection runs only on first chunks (1 call in "
                    "8 of the headline); update chunks project N/4 rows per video"}


def run_single_video(dev, reps=200):
    """Latency view of BASELINE cfg2 read literally (ONE video, chunks strictly sequential): an update call
    captured once as a CUDA graph (5 launches) and replayed.  Launch/latency-bound by construction; throughput
    comes from batching videos (the headline)."""
    from infinite_video_b200.batched import BatchedRectLTM
    torch.manual_seed(0)
    key, val = torch.nn.Linear(E, D), torch.nn.Linear(E, D)
    eng = BatchedRectLTM(NB, TAU, key.weight.detach(), key.bias.detach(), val.weight.detach(), val.bias.detach(),
                         tokens_per_frame=T, device=dev)
    g = torch.Generator(device=dev).manual_seed(7)
    k = torch.randn(1, L * T, E, device=dev, generator=g)
    q = torch.randn(1, Q, D, device=dev, generator=g)
    u = torch.rand(1, S, device=dev, dtype=torch.float64, generator=g)
    eng.step(k, q, None, new_doc=True)
    side = torch.cuda.Stream(device=dev)
    side.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(side):
        eng.step(k, q, u, new_doc=False)
        eng.step(k, q, u, new_doc=False)
    torch.cuda.current_stream(dev).wait_stream(side)
    graphs = []
    for _ in range(2):                       # the coefficient buffers ping-pong: one graph per parity
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr):
            eng.step(k, q, u, new_doc=False)
        graphs.append(gr)
    for i in range(10):
        graphs[i & 1].replay()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(dev)
    e0.record()
    for i in range(reps):
        graphs[i & 1].replay()
    e1.record()
    torch.cuda.synchronize(dev)
    us_call = 1e3 * e0.elapsed_time(e1) / reps
    return {"videos": 1, "us_per_call": us_call, "value": 1e6 / us_call, "unit": "chunks/s",
            "note": "one video, CUDA-graph replay of a sticky update call (k re-read from L2: 25 MB < 126 MB L2)"}


_JSON_OUT = None


def claim_stdout():
    """stdout carries exactly one JSON line: keep a private handle to it and point fd 1 at stderr for the rest of
    the run, so that library banners written by native code (NCCL prints its version at communicator creation)
    cannot precede or follow the line."""
    global _JSON_OUT
    if _JSON_OUT is None:
        sys.stdout.flush()
        _JSON_OUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line):
    out = _JSON_OUT if _JSON_OUT is not None else sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--videos", type=int, default=128, help="videos per GPU (weak scaling)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: --videos per GPU; strong: --total-videos sharded over the GPUs (BASELINE configs[4])")
    ap.add_argument("--total-videos", type=int, default=1024)
    ap.add_argument("--chunks", type=int, default=8, help="sequential chunks per video")
    ap.add_argument("--precision", default="tf32", choices=["tf32", "tf32x3"])
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-overlap", action="store_true", help="do not pool chunk c+1 under chunk c's compute")
    ap.add_argument("--pool-ctas-per-sm", type=int, default=0, help="grid bound of the prefetch pooling kernel")
    ap.add_argument("--proj-operands", choices=["fp32", "fp16"], default="fp16",
                    help="operands of the K/V projection on the tensor-core path (fp16: kind::f16 UMMAs, opt-in)")
    ap.add_argument("--kv-dtype", default="fp16", choices=["fp32", "fp16"],
                    help="storage of the projected memory K|V on the tensor-core path")
    ap.add_argument("--no-bin-pool", action="store_true",
                    help="pool every frame on its own (round-1 layout) instead of one row per basis bin on update chunks")
    ap.add_argument("--gemm-ctas", type=int, default=None,
                    help="grid bound of the K/V projection while the next chunk is pooled beside the step "
                         "(default: the engine's 7/16 of the SMs; 0 = one CTA per SM)")
    ap.add_argument("--video-block", type=int, default=0,
                    help="consolidate / project / attend in blocks of this many videos (L2 reuse); 0 = all at once")
    ap.add_argument("--no-kv-state", action="store_true",
                    help="project all N coefficient rows every call instead of carrying K|V of the old bins along")
    ap.add_argument("--proj-precision", default=None, choices=["tf32", "tf32x3"],
                    help="precision of the K/V projection GEMM alone (default: --precision)")
    ap.add_argument("--repeats", type=int, default=3, help="timed regions of K steps each; the fastest is reported")
    ap.add_argument("--graph", action="store_true",
                    help="also time the K steps replayed from one CUDA graph per step (measured: 160 k vs 175 k eager -- "
                         "the host needs 0.8 ms to enqueue a 5.9 ms step, and graph kernel nodes lose the stream priorities)")
    ap.add_argument("--hi-prio", action="store_true", help="run the main stream at high priority")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gauss", action="store_true", help="skip the secondary Gaussian-variant measurement")
    ap.add_argument("--sustain-s", type=float, default=2.0,
                    help="length of the additional sustained timed region in seconds (0 = skip)")
    ap.add_argument("--no-configs", action="store_true", help="skip the other BASELINE shapes (cfg1 / cfg3 / cfg4)")
    ap.add_argument("--gauss-videos", type=int, default=128)
    ap.add_argument("--gauss-frames", type=int, default=256, help="Lk of the Gaussian arm (k is consumed un-pooled)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the contexts the last timed step returned as DIR/ctx_chunk<c>.npy (float32 [videos,Q,D]"
                         "; a fixed seeded sample of the videos when all would exceed 64 MB), for comparing two builds")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.impl == "reference":
        return run_reference_impl(args)
    if args.hi_prio:
        with torch.cuda.stream(torch.cuda.Stream(priority=-1)):
            return run_b200(args)
    return run_b200(args)


if __name__ == "__main__":
    sys.exit(main())
