"""LTM consolidation for Bv independent videos with explicit per-video state and explicit uniforms.

This is the layer the reference does not have: its module is batch-1 and sequential
(long_term_attention_gibbs.py:346 `reshape(1, qlen, -1)`, :208 `ts[0]`).  Chunks of one video stay strictly
sequential (B_past and the sticky density depend on the previous call), videos are independent, so the
batch dimension is the only free axis and every kernel carries it.

State per video
  variant R: B_past[N,e]; sticky histogram partials of the previous call's density [H*ceil(Q/32),127]
  variant G: B_past[N,e]; (mu, sigma)[H*Q] of the previous call
"""
import ctypes as C
import functools
import math
import weakref

import numpy as np
import torch

from . import ops, tables
from ._capi import Overlap, RectStepArgs, check, lib, ptr, require_cuda, stream_ptr

@functools.lru_cache(maxsize=None)
def _sm_count(index):
    return torch.cuda.get_device_properties(index).multi_processor_count


def _on_device(fn):
    """Run a method with the engine's device current: the library launches on the stream handle it is given, and
    handles of one device are invalid while another device is current (a model sharded over several GPUs of one
    process)."""
    @functools.wraps(fn)
    def wrapped(self, *a, **kw):
        if torch.cuda.current_device() == self.device.index:
            return fn(self, *a, **kw)
        with torch.cuda.device(self.device):
            return fn(self, *a, **kw)
    return wrapped


def _as_flags(new_doc, Bv, device):
    """bool | sequence | tensor -> (all_new: bool|None, uint8 device tensor|None)."""
    if isinstance(new_doc, (bool, int)):
        return bool(new_doc), None
    t = torch.as_tensor(new_doc)
    if t.numel() != Bv:
        raise ValueError("new_doc must be a bool or one flag per video")
    t = t.to(device=device, dtype=torch.uint8).contiguous()
    return None, t


def _as_lengths(lengths, Bv, Lmax):
    """Per-video chunk lengths of a ragged step -> int tuple; 0 (idle) or within [2, Lmax].  Host values only: the
    tables are selected from them on the host, and reading a CUDA tensor would be a hidden synchronisation."""
    if isinstance(lengths, torch.Tensor):
        if lengths.device.type != "cpu":
            raise ValueError("lengths must be host integers (a list or a CPU tensor), not a CUDA tensor")
        if lengths.is_floating_point() or lengths.is_complex():
            raise ValueError("lengths must be integers")
        lengths = lengths.reshape(-1).tolist()
    vals = tuple(int(x) for x in lengths)
    if any(float(x) != float(y) for x, y in zip(vals, lengths)):
        raise ValueError("lengths must be integers")
    if len(vals) != Bv:
        raise ValueError(f"lengths must hold one value per video ({Bv}), got {len(vals)}")
    for x in vals:
        if x != 0 and not 2 <= x <= Lmax:
            raise ValueError(f"chunk length {x} is outside [2, {Lmax}] (0 = idle; chunks of one frame are not "
                             "supported)")
    return vals


class _Entries:
    """A chunk given per video (see `BatchedRectLTM.step`), validated: the entries (None = idle), their lengths in
    frames, the storage code of the present ones, their base addresses, one entry per distinct storage (the tensors to
    `record_stream` on a stream that reads them) and `shape` = (Bv, L*T, e), the padded chunk it stands for."""
    __slots__ = ("entries", "lens", "code", "ptrs", "stores", "shape")


def _chunk_refs(k):
    """Identity of a chunk for prefetch matching: per tensor (one for a padded chunk, one per entry of a list) a weak
    reference and its version counter.  A data pointer is not a key: the caching allocator hands the same address to
    the next chunk, and an in-place write changes the contents behind an unchanged pointer."""
    ts = k.entries if isinstance(k, _Entries) else (k,)
    return tuple(None if t is None else (weakref.ref(t), t._version) for t in ts)


def _refs_match(refs, k):
    ts = k.entries if isinstance(k, _Entries) else (k,)
    return len(refs) == len(ts) and all(
        (t is None) if r is None else (t is not None and r[0]() is t and r[1] == t._version) for r, t in zip(refs, ts))


def _refs_alive(refs):
    return all(r is None or r[0]() is not None for r in refs)


def _pad_rows(m):
    """Copy a 2-D matrix into storage whose row pitch is a multiple of 4 floats (TMA: 16-byte pitches)."""
    r, c = m.shape
    buf = torch.zeros(r, (c + 3) // 4 * 4, device=m.device, dtype=torch.float32)
    buf[:, :c] = m
    return buf[:, :c]


class _BatchedBase:
    def __init__(self, num_basis, tau, w_key, b_key, w_value, b_value, n_heads, head_size, sticky, nb_samples,
                 precision, device):
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise ValueError("the LTM consolidation path runs on CUDA devices only (no CPU fallback)")
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.sm_count = _sm_count(self.device.index)
        self.N = int(num_basis)
        self.tau = float(tau)
        self.H, self.d = int(n_heads), int(head_size)
        self.D = self.H * self.d
        self.sticky = bool(sticky)
        self.S = int(nb_samples)
        self.precision = precision
        self.gemm_impl = "tcgen05"      # one backend: the SIMT GEMM is a kernel-level test cross-check (ops.gemm impl=)
        self.set_projections(w_key, b_key, w_value, b_value)
        self.Bv = None
        self.has_state = False

    def set_projections(self, w_key, b_key, w_value, b_value):
        """[W_key ; W_value] -> one [2D,e] operand so K and V come out of a single GEMM (gibbs:312-313)."""
        dev = self.device
        wk = w_key.detach().to(dev, torch.float32)
        wv = w_value.detach().to(dev, torch.float32)
        self.e = wk.shape[1]
        if wk.shape[0] != self.D or wv.shape != wk.shape:
            raise ValueError(f"projection weights must be [{self.D}, e]")
        bk = torch.zeros(self.D, device=dev) if b_key is None else b_key.detach().to(dev, torch.float32)
        bv = torch.zeros(self.D, device=dev) if b_value is None else b_value.detach().to(dev, torch.float32)
        self.Wkv = torch.cat([wk, wv], 0).contiguous()
        self.bkv = torch.cat([bk, bv], 0).contiguous()

    def reset(self):
        """Forget every video (new_doc for all)."""
        self.has_state = False


class BatchedRectLTM(_BatchedBase):
    """Variant R ("gibbs", the live module): rectangular bases, Gibbs density.
    One `step` == one `LongTermAttention.forward` per video (gibbs:288-346)."""

    def __init__(self, num_basis, tau, w_key, b_key, w_value, b_value, *, n_heads=12, head_size=64,
                 tokens_per_frame=32, sticky=True, nb_samples=tables.NB_SAMPLES, precision="tf32",
                 device="cuda", keep_scores=False, fast_attn=True, tc_attn=True,
                 proj_operands="fp16", kv_state=True, proj_precision=None, spacing="linear", kv_dtype="fp16",
                 bin_pool=None):
        super().__init__(num_basis, tau, w_key, b_key, w_value, b_value, n_heads, head_size, sticky, nb_samples,
                         precision, device)
        self.T = int(tokens_per_frame)
        # frame pooling folded with the regression of update chunks (csrc/pool.cu: pool_bins_kernel): the pooling
        # kernel writes one row per basis bin (the sum of the pooled frames that fall into it) instead of one per
        # frame.  None: when it pays (three or more frames per bin, enough (video, bin) pairs to fill the GPU); True: whenever
        # the tables allow it; False: never.  Applies where this engine pools the chunk itself (`step` without
        # `pooled=`, `prefetch(update=True)`, `step_overlapped`).
        self.bin_pool = bin_pool
        # grid bound of the K/V projection while the next chunk is pooled beside the step (0 = all SMs): the projection
        # is not on the critical path there, and on 64 of the 148 SMs it takes less of the L2 -> SM bandwidth the
        # pooling kernel needs at any one time (step 194.6 k -> 207.3 k chunks/s; 32 .. 77 CTAs within 1 % of each other)
        self.gemm_ctas_overlap = max(32, (self.sm_count * 7) // 16)
        self.gemm_ctas_min_ratio = 16          # chunk tokens per basis function from which the bound applies
        self.spacing = spacing        # first-chunk frame positions: 'linear' | 'log' (gibbs:101-127)
        self.keep_scores = keep_scores
        # transposed-key attention path (num_basis 64/128/256, head size 64); `fast_attn=False` forces the generic one
        self.fast_attn = bool(fast_attn) and ops.attn_fast_supported(self.N, self.d)
        # tensor-core attention (csrc/attn_tc.cu): num_basis 64/128/256, head size 64, single-pass tf32 projection
        # (num_basis 512: the same kernel over the two halves of the basis range + a combine kernel)
        self.tc_split = ops.attn_tc_split_supported(self.N, self.d)
        self.tc_attn = (bool(tc_attn) and bool(fast_attn) and precision == "tf32"
                        and (ops.attn_tc_supported(self.N, self.d) or self.tc_split))
        self.tc_split = self.tc_split and self.tc_attn
        # operands of the K/V projection on the tensor-core path: "fp16" (default) -- the consolidation also writes the
        # coefficient rows the projection will read as fp16 (round to nearest: unbiased, where the tensor core
        # TRUNCATES fp32 operands read as tf32) and the weights are kept as fp16: kind::f16 UMMAs at twice the TF32
        # rate and half the operand bytes (projection 0.064 -> 0.040 ms per 128-video chunk, 190.3 k -> 193.5 k
        # chunks/s) -- or "fp32" (tf32 UMMAs straight from the fp32 tensors).  fp16's range applies: |B|, |W| <= 65504.
        if proj_operands not in ("fp16", "fp32"):
            raise ValueError("proj_operands must be 'fp16' or 'fp32'")
        self.half_ops = self.tc_attn and proj_operands == "fp16" and self.e % 8 == 0
        # projected-memory state (csrc/consolidate.cu): K|V = B W^T + b is affine in B and the memory contraction is
        # linear, so K|V of the bins that hold only re-sampled memory are the same segmented mean taken over the
        # previous K|V; only the bins that receive new frames (a quarter at tau = 0.75) go through the projection GEMM.
        # Needs the row-major K|V layout (tensor-core or generic attention) and one new_doc flag for the whole batch.
        self.kv_state = bool(kv_state) and (self.tc_attn or not self.fast_attn)
        # precision of the K/V projection GEMM alone (None = `precision`); "tf32x3" makes the stored K|V fp32-grade
        self.proj_precision = proj_precision
        # storage of the projected memory on the tensor-core path: "fp16" (default) or "fp32" (values on the tf32
        # grid).  fp16 carries the same 11-bit significand as that grid at half the bytes -- K|V are written once and
        # read twice per call: ~250 MB less per 128-video chunk, 181.0 k -> 190.0 k chunks/s -- and the attention
        # contractions run as kind::f16 UMMAs.  What it gives up is range: |K|, |V| > 65504 become inf (and show up as
        # NaN contexts); keys / values are projections of layer-normed features, orders of magnitude below that, and
        # the VideoChat2 pipeline of the reference computes them in fp16 itself (autocast).
        if kv_dtype not in ("fp32", "fp16"):
            raise ValueError("kv_dtype must be 'fp32' or 'fp16'")
        self.kv_half = kv_dtype == "fp16" and self.tc_attn
        self._Wkv_h = None
        self.prof_events = None       # optional list of 10 cudaEvent_t handles (bench.py stage timing)
        self._side = None             # side stream for pooling the next chunk ahead of time
        self._pref = []               # pending prefetches, oldest first (see `prefetch`)
        self._evs = None              # persistent fork / join events of the two-stream schedule
        self.pool_ctas = 0            # grid bound of the side-stream pooling kernel (0 = one CTA per frame)
        self._ws = {}
        self._B = None
        self._cur = 0
        self.last = {}
        self._slots = None            # per-slot memory after ragged steps (bool [Bv]); None: every slot has_state
        self._banks = {}              # Lmax -> tables.RectBank
        self._last_ragged = False

    # ------------------------------------------------------------------ buffers
    def _workspace(self, Bv, L, Q):
        key = (Bv, L, Q)
        ws = self._ws.get(key)
        if ws is None:
            dev = self.device
            units = Bv * L
            # split the token range of a frame over several CTAs only when there are too few frames to fill the
            # 148 SMs (small batches); otherwise one CTA per frame, one pass, no partial sums
            splits = self._splits(units)
            f32 = dict(device=dev, dtype=torch.float32)
            i32 = dict(device=dev, dtype=torch.int32)
            # pooled-frame buffers: [Bv, L, splits, e] per-frame partial means, or -- same storage -- [Bv, rows, e]
            # per-bin sums (xtag[i]: what buffer i currently holds)
            xrows = max(L * splits, self.N)
            xbufs = [torch.empty(Bv * xrows * self.e, **f32) for _ in range(2)]
            ws = dict(
                splits=splits,
                xbufs=xbufs,
                xparts=[b[:Bv * L * splits * self.e].view(Bv, L, splits, self.e) for b in xbufs],
                xtag=[False, False],
                xi=0,
                KVs=[torch.empty(Bv, self.N, 2 * self.D, device=dev,
                                 dtype=torch.float16 if self.kv_half else torch.float32)
                     for _ in range(2 if self.kv_state else 1)]
                if (self.tc_attn or not self.fast_attn) else None,
                Kt=torch.empty(Bv, self.H, self.d, self.N, **f32) if (self.fast_attn and not self.tc_attn) else None,
                V=torch.empty(Bv, self.N, self.D, **f32) if (self.fast_attn and not self.tc_attn) else None,
                b_draw=torch.empty(Bv, self.S, **i32), idx=torch.empty(Bv, self.S, **i32),
                ts=torch.empty(Bv, self.S, **f32), p=torch.empty(Bv, 127, **f32),
                scores=torch.empty(Bv, self.H, Q, self.N, **f32) if (self.keep_scores or self.tc_split) else None,
                attn_part=torch.empty(int(lib().ltm_attn_tc_split_workspace_floats(Bv, Q, self.H)), **f32)
                if self.tc_split else None,
                B_half=torch.empty(Bv, self.N, self.e, device=dev, dtype=torch.float16) if self.half_ops else None,
                k_dev=None, q_dev=None, u_dev=None, nd_dev=None, ctx_dev=None,
            )
            self._ws = {key: ws}          # one live shape at a time
        return ws

    def _splits(self, units):
        """Token-splits of the frame pooling: one CTA per frame when that already gives the GPU four waves of CTAs
        (8 resident per SM), otherwise each frame's tokens are split so that it does -- a grid of barely more than one
        wave leaves the second one almost empty (VideoChat2 shape, 64 videos x 16 frames = 1024 CTAs for 1184 slots:
        146 us for 822 MB).  No units (a ragged chunk of idle videos): 1."""
        want = 4 * 8 * self.sm_count
        # (at most T/8 splits: the partial sums are written and read back, T/splits rows of input per row of output)
        return 1 if units >= want or units == 0 else max(1, min(max(1, self.T // 8), -(-want // units)))

    def _bin_ok(self, Bv, L, tab, k_dtype=0):
        """Whether an update chunk of this shape and storage (k_dtype, see `_chunk_dtype`) is pooled per bin (see
        `bin_pool`).  A 16-bit chunk never is: it is pooled per frame, as `step` always pooled it."""
        if k_dtype or self.bin_pool is False or tab.xb_rows <= 0:
            return False
        if self.bin_pool:
            return True
        # (measured: 4 frames per bin +0.4 % burst / +1.1 % sustained at the NExT-QA shape; 2 per bin -2 % at num_basis 512)
        return L >= 3 * tab.xb_rows and Bv * tab.xb_rows >= 4 * 8 * self.sm_count

    def _chunk_dtype(self, k, name="k"):
        """Storage code of chunk k (0 float32, 1 float16, 2 bfloat16); ValueError for any other dtype, and for a 16-bit
        chunk whose width is not a multiple of 8 (it is read as 128-bit vectors of 8 elements)."""
        dt = ops.CHUNK_DTYPES.get(k.dtype)
        if dt is None:
            raise ValueError(f"{name} must be float32, float16 or bfloat16, not {k.dtype}")
        if dt and k.shape[-1] % 8:
            raise ValueError(f"a 16-bit {name} needs a width that is a multiple of 8, not {k.shape[-1]}")
        return dt

    def _entries(self, k, chunk_frames, lengths=None, name="k"):
        """A chunk given as a list of Bv entries (see `step`) -> `_Entries`; a tensor (or an `_Entries`) is returned
        as it is.  Every entry is checked before any state changes, and nothing is copied: a silent `.contiguous()`
        would bring back the copy this form exists to avoid, and break prefetch matching."""
        if not isinstance(k, (list, tuple)):
            if chunk_frames is not None and not isinstance(k, _Entries):
                raise ValueError(f"chunk_frames applies to a chunk given as a list, and {name} is a tensor")
            return k
        if lengths is not None:
            raise ValueError(f"{name} given as a list carries its own lengths: do not pass lengths as well")
        if chunk_frames is None:
            raise ValueError(f"{name} given as a list needs chunk_frames= (the padded chunk length L)")
        L, T, e = int(chunk_frames), self.T, self.e
        if L < 2 or not k:
            raise ValueError(f"{name} given as a list needs chunk_frames >= 2 and at least one entry")
        lens, ptrs, stores, dtype = [], [], {}, None
        for v, t in enumerate(k):
            if t is None:
                lens.append(0)
                ptrs.append(0)
                continue
            if not isinstance(t, torch.Tensor) or t.device != self.device:
                raise ValueError(f"{name}[{v}] must be None or a tensor on {self.device}")
            if dtype is None:
                dtype = t.dtype
                code = self._chunk_dtype(t, f"{name}[{v}]")
            elif t.dtype != dtype:
                raise ValueError(f"{name}[{v}] is {t.dtype}, the entries before it {dtype}: one dtype per chunk")
            if t.dim() != 2 or t.shape[1] != e:
                raise ValueError(f"{name}[{v}] must be [n*{T}, {e}], not {list(t.shape)}")
            n = t.shape[0]
            if n % T or not 2 <= n // T <= L:
                raise ValueError(f"{name}[{v}] has {n} tokens: a multiple of {T} for 2 to {L} frames (None = idle)")
            if t.stride() != (e, 1):
                raise ValueError(f"{name}[{v}] must have dense rows, strides ({e}, 1), not {t.stride()}")
            p = t.data_ptr()
            if p % 16:
                raise ValueError(f"{name}[{v}] must start at a 16-byte aligned address")
            lens.append(n // T)
            ptrs.append(p)
            stores.setdefault(t.untyped_storage().data_ptr(), t)
        c = _Entries()
        c.entries, c.lens, c.code, c.ptrs = tuple(k), tuple(lens), (code if dtype is not None else 0), ptrs
        c.stores, c.shape = tuple(stores.values()), (len(k), L * T, e)
        return c

    def reset(self):
        """Forget every video (new_doc for all) and every pending prefetch."""
        super().reset()
        self._slots = None
        self._pref.clear()

    def cancel_prefetch(self):
        """Drop the chunks pooled ahead of time that were never consumed by a `step`."""
        self._pref.clear()

    # pending prefetches are identified by the tensor OBJECTS (weak references) and their version counters
    # (`_chunk_refs`), and by the lengths
    def _pref_take(self, k, lens=None):
        for i, ent in enumerate(self._pref):
            if ent["lens"] == lens and _refs_match(ent["refs"], k):
                return self._pref.pop(i)
        return None

    def _pref_buffer(self, ws):
        """Buffer for the next prefetch: one that no pending prefetch holds, preferably not the one the most recent
        step consumes.  An abandoned prefetch (tensor gone, or never stepped) is evicted, oldest first."""
        self._pref[:] = [e for e in self._pref if _refs_alive(e["refs"])]
        while len(self._pref) >= 2:
            self._pref.pop(0)
        held = {e["buf"] for e in self._pref}
        pref = 1 - ws["xi"]
        return pref if pref not in held else 1 - pref

    def _frames_source(self, k, Q, ws, tab, flags, rag, pooled=None, prefetch=False):
        """Where the pooled frames of chunk k come from, for `step` and `step_overlapped`: `pooled` when given (returns
        None); else a pending prefetch of k, whose entry is returned with ws["xi"] on its buffer; else, with
        `prefetch`, one issued here; else the step pools k itself (returns None), into a buffer that no pending
        prefetch holds."""
        if pooled is not None:
            return None
        lens = None if rag is None else rag["lens"]
        update = rag is None and self.has_state and flags is None   # every video continues: per-bin pooling possible
        hit = self._pref_take(k, lens)
        if hit is not None and hit["binned"] and not update:
            hit = None                                   # pooled per bin for an update that did not come: pool again
        if hit is None and prefetch:
            if isinstance(k, _Entries):
                self.prefetch(k, Q)
            else:
                self.prefetch(k, Q, lengths=lens, update=update)
            hit = self._pref_take(k, lens)
        if hit is not None:
            ws["xi"] = hit["buf"]
            ws["xtag"][hit["buf"]] = hit["binned"]
            return hit
        held = {e["buf"] for e in self._pref}          # never pool over frames a pending prefetch still owns
        ws["xi"] = (1 - ws["xi"]) if (1 - ws["xi"]) not in held else ws["xi"]
        if ws["xi"] in held:
            self._pref[:] = [e for e in self._pref if e["buf"] != ws["xi"]]
        ws["xtag"][ws["xi"]] = update and self._bin_ok(k.shape[0], k.shape[1] // self.T, tab,
                                                       ops.CHUNK_DTYPES.get(k.dtype, 0))
        return None

    def _state(self, Bv, Q):
        qt = (Q + 31) // 32
        if self._B is None or self.Bv != Bv or self._hist.shape[1] != self.H * qt:
            f32 = dict(device=self.device, dtype=torch.float32)
            self._B = [torch.zeros(Bv, self.N, self.e, **f32), torch.zeros(Bv, self.N, self.e, **f32)]
            self._hist = torch.ones(Bv, self.H * qt, 127, **f32)
            self._cur = 0
            self.Bv = Bv
            self.has_state = False
            self._slots = None

    @property
    def B_past(self):
        return self._B[self._cur] if (self._B is not None and self.has_state) else None

    # ------------------------------------------------------------------ one chunk
    def _args(self, Bv, L, Q, ws, tab, tdev, beside_pool=False, rag=None, k_dtype=0):
        # the argument block is built once per workspace / table set / weights and only its per-call fields are
        # rewritten afterwards (the ~40 ctypes assignments were a third of the host time of a chunk)
        sig = (id(tdev), self.Wkv.data_ptr(), self.bkv.data_ptr(), self._hist.data_ptr(), self.sticky,
               self.precision, self.gemm_impl, ws["k_dev"] is None)
        a = ws.get("_args")
        if a is None or ws.get("_args_sig") != sig:
            a = self._args_full(Bv, L, Q, ws, tab, tdev)
            ws["_args"], ws["_args_sig"], ws["_args_prof"] = a, sig, False
            ws["_args_keep"] = (tdev, self.Wkv, self.bkv, self._hist)     # the block holds raw pointers into these
        a.splits = ws["splits"]
        a.B_past = self._B[self._cur].data_ptr() if self.has_state else None
        a.B_new = self._B[1 - self._cur].data_ptr()
        a.xpart = ws["xbufs"][ws["xi"]].data_ptr()
        a.binned = 1 if ws["xtag"][ws["xi"]] else 0
        a.k_dtype, a.k_ptrs = k_dtype, None
        # (only where the pooling is the long pole of the step: a chunk of at least 16 tokens per basis function; with
        # 8 frames x 32 tokens on 64 bins the chain of this stream is, and a narrower projection would lengthen it)
        bound = beside_pool and L * self.T >= self.gemm_ctas_min_ratio * self.N
        a.gemm_ctas = int(self.gemm_ctas_overlap) if bound else 0
        if ws["KVs"] is not None and len(ws["KVs"]) == 2:      # K|V ping-pong, in phase with the coefficient buffers
            a.KV = ws["KVs"][1 - self._cur].data_ptr()
            a.KV_past = ws["KVs"][self._cur].data_ptr() if (self.has_state and ws.get("kv_valid")) else None
        if rag is None:
            a.lengths, a.frame_offs, a.n_idle, a.jf = None, None, 0, tab.jf
        else:
            bank = rag["bank"]
            a.lengths, a.frame_offs = rag["lens_dev"].data_ptr(), rag["offs_dev"].data_ptr()
            a.frames, a.n_idle, a.jf, a.splits, a.binned = rag["frames"], rag["n_idle"], rag["jf"], rag["splits"], 0
            a.bank_seg_ptr0, a.bank_seg_mem0, a.bank_g0 = (bank["seg_ptr0"].data_ptr(), bank["seg_mem0"].data_ptr(),
                                                           bank["g0"].data_ptr())
            a.bank_seg_ptr1, a.bank_seg_mem1, a.bank_g1 = (bank["seg_ptr1"].data_ptr(), bank["seg_mem1"].data_ptr(),
                                                           bank["g1"].data_ptr())
            a.hist_keep = rag["hist_keep"].data_ptr() if rag["hist_keep"] is not None else None
        if self.prof_events is not None:
            for i, ev in enumerate(self.prof_events):
                a.prof_events[i] = ev
            ws["_args_prof"] = True
        elif ws["_args_prof"]:
            for i in range(10):
                a.prof_events[i] = None
            ws["_args_prof"] = False
        return a

    def _args_full(self, Bv, L, Q, ws, tab, tdev):
        a = RectStepArgs()
        a.Bv, a.L, a.T, a.e, a.N, a.Q, a.H, a.d, a.S = Bv, L, self.T, self.e, self.N, Q, self.H, self.d, self.S
        a.splits, a.sticky = ws["splits"], int(self.sticky)
        a.precision, a.gemm_impl = ops.PRECISION[self.precision], ops.GEMM_IMPL[self.gemm_impl]
        for name in ("seg_ptr0", "seg_mem0", "g0", "seg_ptr1", "seg_mem1", "g1", "jb", "tb", "bins", "bin2basis",
                     "idx_uniform", "W"):
            setattr(a, name, tdev[name].data_ptr())
        a.W_out = tab.W_out
        if self.tc_attn:
            if tdev["X"] is None:
                raise RuntimeError("tensor-core attention needs a quadrature point in every basis (tc_attn=False)")
            a.X, a.c_none = tdev["X"].data_ptr(), tab.c_none
        a.Wkv, a.bkv = self.Wkv.data_ptr(), self.bkv.data_ptr()
        if self.half_ops:
            if self._Wkv_h is None or self._Wkv_h_src != self.Wkv.data_ptr():
                self._Wkv_h, self._Wkv_h_src = self.Wkv.to(torch.float16).contiguous(), self.Wkv.data_ptr()
            a.B_half, a.Wkv_half = ws["B_half"].data_ptr(), self._Wkv_h.data_ptr()
        a.B_past = self._B[self._cur].data_ptr() if self.has_state else None
        a.B_new = self._B[1 - self._cur].data_ptr()
        a.hist_part = self._hist.data_ptr()
        a.xpart = ws["xbufs"][ws["xi"]].data_ptr()
        if tab.xb_rows > 0:
            a.xb_rows = tab.xb_rows
            a.fbin_ptr, a.seg_ptr1b, a.seg_mem1b = (tdev["fbin_ptr"].data_ptr(), tdev["seg_ptr1b"].data_ptr(),
                                                    tdev["seg_mem1b"].data_ptr())
        a.KV = ws["KVs"][0].data_ptr() if ws["KVs"] is not None else None
        a.KV_past = None
        a.jf = tab.jf
        a.proj_precision = ops.PRECISION[self.proj_precision] if self.proj_precision else 0
        a.Kt = ws["Kt"].data_ptr() if ws["Kt"] is not None else None
        a.V = ws["V"].data_ptr() if ws["V"] is not None else None
        a.b_draw, a.idx, a.ts, a.p = (ws["b_draw"].data_ptr(), ws["idx"].data_ptr(), ws["ts"].data_ptr(),
                                      ws["p"].data_ptr())
        a.scores = ws["scores"].data_ptr() if ws["scores"] is not None else None
        a.attn_part = ws["attn_part"].data_ptr() if ws["attn_part"] is not None else None
        if self.kv_half:
            a.kv_half, a.X16 = 1, tdev["X16"].data_ptr()
        for f, n in (("k_dev", "k_dev"), ("q_dev", "q_dev"), ("u_dev", "u_dev"), ("new_doc_dev", "nd_dev"),
                     ("ctx_dev", "ctx_dev")):
            setattr(a, f, ws[n].data_ptr() if ws[n] is not None else None)
        return a

    def _prepare(self, k, q, new_doc, u, lengths=None, pooled=None, u_name="u", ptrs=None):
        """Host side of a step: validation, per-slot bookkeeping, tables.  Every ValueError fires before any state
        changes.  Returns (Bv, L, Q, tab, tdev, flags, u, rag): the device new_doc flags the step applies (None: none),
        the contiguous uniforms (None: the step reads none) and, for a ragged step, its table bank and device lengths /
        offsets (rag; None: lock-step).  A lock-step call takes new_doc as a device tensor too, a ragged one as host
        flags (it selects tables from them)."""
        if getattr(self, "video_block", 0):
            # the step in blocks of videos (4-14 % slower at every block size) was removed; refusing the setting keeps
            # a caller from running, and recording, a block size that has no effect
            raise ValueError("video_block: the blocked step was removed; every kernel covers all videos")
        Bv, LT, e = k.shape
        if e != self.e:
            raise ValueError(f"k has width {e}, projections expect {self.e}")
        if lengths is None and LT % self.T:
            raise ValueError(f"k has {LT} tokens, not a multiple of tokens_per_frame={self.T}")
        if lengths is not None and (LT % self.T or LT // self.T < 2):
            raise ValueError(f"k has {LT} tokens: a ragged chunk is padded to L*{self.T} tokens, L >= 2")
        L, Q = LT // self.T, q.shape[1]
        if q.shape[0] != Bv or q.shape[2] != self.D:
            raise ValueError(f"q must be [{Bv}, Q, {self.D}]")
        same = self.has_state and self._B is not None and self.Bv == Bv        # this batch has memory to continue
        # the sticky histogram of the previous call is kept per (head, tile of 32 queries): a different number of
        # query tiles inside a video would silently restart the memory
        retiled = same and self._hist.shape[1] != self.H * ((Q + 31) // 32)
        retiled_msg = f"the number of queries changed inside a video ({Q} now): pass new_doc=True or keep Q"
        if lengths is None:
            all_new, flags = _as_flags(new_doc, Bv, self.device)
            keep = same and not all_new
            if keep and retiled:
                raise ValueError(retiled_msg)
            if keep and self._slots is not None and not self._slots.all():
                # (only after a ragged step left slots without memory)
                nd = torch.as_tensor(new_doc).reshape(-1).to("cpu", torch.bool).numpy() if all_new is None else False
                self._no_memory_check(~np.asarray(nd, bool) & ~self._slots)
            need_u = keep and self.sticky
        else:
            ln = np.asarray(_as_lengths(lengths, Bv, L), np.int64)
            if isinstance(new_doc, (bool, int)):
                nd = np.full(Bv, bool(new_doc))
            else:
                t = torch.as_tensor(new_doc)
                if t.device.type != "cpu" or t.numel() != Bv:
                    raise ValueError("a ragged step takes new_doc as a bool or one host flag per video")
                nd = t.reshape(-1).to(torch.bool).numpy()
            present = ln > 0
            mem = (self._slots if self._slots is not None else np.ones(Bv, bool)) if same else np.zeros(Bv, bool)
            if retiled and (mem & ~nd).any():
                raise ValueError(retiled_msg)
            cont = present & ~nd
            self._no_memory_check(cont & ~mem)
            keep = same and not retiled
            need_u = keep and self.sticky and bool(cont.any())
            frames = int(ln.sum())
            if pooled is not None and (pooled.dim() != 3 or pooled.shape[0] != frames or pooled.shape[2] != self.e):
                raise ValueError(f"pooled frames of a ragged chunk must be [{frames}, splits, {self.e}]")
        if pooled is not None and (not pooled.is_contiguous() or lengths is None and (
                tuple(pooled.shape[:2]) != (Bv, L) or pooled.shape[3] != self.e)):
            raise ValueError("pooled frames do not match k")
        if need_u:
            if u is None or u.dtype != torch.float64 or tuple(u.shape) != (Bv, self.S):
                raise ValueError(f"sticky re-sampling needs {u_name}: float64 [{Bv},{self.S}]")
            u = u.contiguous()
        else:
            u = None
        self._state(Bv, Q)
        self.has_state = keep                # False: every video starts with this chunk
        tab = tables.rect_tables(L, self.N, self.tau, self.S, spacing=self.spacing)
        if lengths is None:
            return Bv, L, Q, tab, tab.to(self.device), flags if keep else None, u, None
        first = present & nd
        flags = None
        if keep and first.any():
            flags = torch.from_numpy(first.astype(np.uint8)).pin_memory().to(self.device, non_blocking=True)
        bank = self._bank(L)
        bdev = bank.to(self.device, set(ln.tolist()))
        n_idle = int((~present).sum())
        hist_keep = None
        if n_idle and self.sticky:
            if getattr(self, "_hist_keep", None) is None or self._hist_keep.shape != self._hist.shape:
                self._hist_keep = torch.empty_like(self._hist)
            hist_keep = self._hist_keep
        lens_dev, offs_dev, ptrs_dev = self._lengths_dev(ln, ptrs)
        rag = dict(lens=tuple(ln.tolist()), lens_dev=lens_dev, offs_dev=offs_dev, ptrs_dev=ptrs_dev, bank=bdev,
                   frames=frames,
                   splits=self._splits(frames), n_idle=n_idle,
                   jf=int(bank.jf[ln[cont]].min()) if (keep and cont.any()) else self.N, hist_keep=hist_keep,
                   slots=np.where(nd, present, mem))
        return Bv, L, Q, tab, tab.to(self.device), flags, u, rag

    def _no_memory_check(self, bad):
        if np.any(bad):
            raise ValueError(f"video slot(s) {np.flatnonzero(bad).tolist()} hold no memory and receive a chunk without "
                             "new_doc: pass new_doc for their first chunk")

    def _bank(self, L):
        bank = self._banks.get(L)
        if bank is None:
            bank = self._banks[L] = tables.RectBank(L, self.N, self.tau, self.S, spacing=self.spacing)
        return bank

    def _lengths_dev(self, lens, ptrs=None):
        """(lengths [Bv], exclusive prefix sum [Bv+1], pointer table [Bv] or None): views of one device buffer, copied
        on the current stream in one upload -- the int64 entry addresses of a list chunk, then the int32 lengths and
        offsets."""
        Bv = len(lens)
        p = 0 if ptrs is None else 2 * Bv
        host = np.zeros(p + 2 * Bv + 1, np.int32)
        if ptrs is not None:
            host[:p].view(np.int64)[:] = ptrs
        host[p:p + Bv] = lens
        np.cumsum(host[p:p + Bv], out=host[p + Bv + 1:])
        t = torch.from_numpy(host).pin_memory().to(self.device, non_blocking=True)
        return t[p:p + Bv], t[p + Bv:], (t[:p] if ptrs is not None else None)

    def _ragged_ws(self, ws, Bv, L):
        """Packed pooled frames of a ragged step take sum(lengths) * splits rows: at most Bv * L (one split) or, when
        the frames alone do not fill the GPU, fewer than twice the `_splits` target.  Grows the frame buffers of a
        workspace once to hold either (pending prefetches into the old buffers are dropped)."""
        need = max(Bv * L, 2 * 4 * 8 * self.sm_count) * self.e
        if ws["xbufs"][0].numel() >= need:
            return
        if self._side is not None:
            for b in ws["xbufs"]:
                b.record_stream(self._side)
        self._pref.clear()
        splits = ws["splits"]
        ws["xbufs"] = [torch.empty(need, device=self.device, dtype=torch.float32) for _ in range(2)]
        ws["xparts"] = [b[:Bv * L * splits * self.e].view(Bv, L, splits, self.e) for b in ws["xbufs"]]
        ws["xtag"] = [False, False]

    def _finish(self, ws, xp=None, k=None, rag=None):
        # pooled frames of this call (for `x_past`); a call that pooled per bin keeps a weak reference to the chunk
        # instead and pools it again on demand
        binned = xp is None and ws["xtag"][ws["xi"]]
        self._last_xpart = xp if xp is not None else (None if binned else ws["xparts"][ws["xi"]])
        self._last_k = weakref.ref(k) if (binned and k is not None) else None
        self._last_updated = self.has_state          # False: the call just made was a first chunk
        self._cur = 1 - self._cur
        self.has_state = True
        self._last_ragged = rag is not None
        if rag is not None:
            self._last_xpart = self._last_k = None
            self._slots = rag["slots"]
            self.has_state = bool(rag["slots"].any())
        else:
            self._slots = None
        self._last_L = ws["xparts"][0].shape[1]
        kv = None
        if ws["KVs"] is not None:
            ws["kv_valid"] = True                       # the buffer just written is the next call's KV_past
            kv = ws["KVs"][self._cur if len(ws["KVs"]) == 2 else 0]
        V = ws["V"] if ws["V"] is not None else kv[:, :, self.D:]
        self.last = dict(b=ws["b_draw"], ts=ws["ts"], idx=ws["idx"], p=ws["p"], scores=ws["scores"], V=V, KV=kv)

    @_on_device
    def prefetch(self, k_next, Q, lengths=None, events=None, update=False, chunk_frames=None):
        """Pool the frames of the NEXT chunk now, on a side stream, into the alternate buffer.
        `update=True`: the chunk will continue every video (no new_doc), so it may be pooled per bin (`bin_pool`); a
        step that turns out to start a new document pools it again.  `lengths`: the chunk is ragged (see `step`); the
        step that consumes it must pass the same lengths, or it is pooled again.

        Frame pooling (gibbs:304) does not depend on the memory state, and it is the HBM-bound 93 % of a
        call's bytes, while regression / projection / attention of the current chunk are compute-bound; issuing
        it one chunk ahead lets the two overlap.  The following `step(k_next, ...)` must pass the same tensor.
        A 16-bit chunk (float16 / bfloat16) is pooled per frame from its own storage, never per bin.
        `k_next` may be a list of per-video entries with `chunk_frames` (see `step`); the step that consumes it must
        be handed the same tensor objects."""
        k_next = self._entries(k_next, chunk_frames, lengths, "k_next")
        lst = isinstance(k_next, _Entries)
        if lst:
            dt, lengths = k_next.code, k_next.lens
        else:
            require_cuda(k_next)
            dt = self._chunk_dtype(k_next, "k_next")
            if not k_next.is_contiguous():
                raise ValueError("prefetch needs a contiguous chunk (the following step must be given the same tensor)")
        Bv, LT, e = k_next.shape
        if e != self.e or LT % self.T:
            raise ValueError(f"k_next must be [Bv, L*{self.T}, {self.e}]")
        L = LT // self.T
        lens = None if lengths is None else _as_lengths(lengths, Bv, L)
        ws = self._workspace(Bv, L, Q)
        offs = table = None
        frames, splits = 0, ws["splits"]
        if lens is not None:
            self._ragged_ws(ws, Bv, L)
            _, offs, table = self._lengths_dev(lens, k_next.ptrs if lst else None)
            frames = sum(lens)
            splits = self._splits(frames)
        if self._side is None:
            # pooling runs at the lowest priority, the compute-bound kernels of `step` on a high-priority stream:
            # the block scheduler then places regression / projection / attention CTAs as soon as resources free
            # up and the streaming kernel fills whatever is left
            self._side = torch.cuda.Stream(device=self.device, priority=0)
            self._compute = torch.cuda.Stream(device=self.device, priority=-1)
        main = torch.cuda.current_stream(self.device)
        ev = self._sync_events()
        b = self._pref_buffer(ws)
        sp = C.c_void_p(self._side.cuda_stream)
        mp = C.c_void_p(main.cuda_stream)
        # fork: the target buffer was last read by work already queued on `main`.  Persistent events (re-recorded
        # every call) instead of torch's wait_stream, which creates and destroys a CUDA event per call: with four of
        # those per chunk-step the host enqueue time of a step varied between 0.9 and 8 ms from run to run
        check(lib().ltm_event_record(ev["fork_pool"][b], mp), "event_record")
        check(lib().ltm_stream_wait_event(sp, ev["fork_pool"][b]), "stream_wait_event")
        for t in (k_next.stores if lst else (k_next,)):
            t.record_stream(self._side)
        if events is not None:
            check(lib().ltm_event_record(events[0], sp), "event_record")
        tab = tables.rect_tables(L, self.N, self.tau, self.S, spacing=self.spacing)
        binned = lens is None and bool(update) and self._bin_ok(Bv, L, tab, dt)
        if offs is not None:
            offs.record_stream(self._side)          # (the table shares its buffer)
        if lst:
            ops.pool_ptrs(table, dt, ws["xbufs"][b], offs, Bv, L, self.T, e, splits, frames, int(self.pool_ctas), sp)
        else:
            ops.pool_into(k_next, ws["xbufs"][b], L, self.T, splits, int(self.pool_ctas), sp, offs=offs, frames=frames,
                          fbin_ptr=tab.to(self.device)["fbin_ptr"] if binned else None, rows=tab.xb_rows)
        if events is not None:
            check(lib().ltm_event_record(events[1], sp), "event_record")
        check(lib().ltm_event_record(ev["pooled"][b], sp), "event_record")
        self._pref.append(dict(refs=_chunk_refs(k_next), buf=b, event=ev["pooled"][b],
                               captured=torch.cuda.is_current_stream_capturing(), binned=binned, lens=lens))

    def _sync_events(self):
        if self._evs is None:
            def mk():
                h = C.c_void_p()
                check(lib().ltm_event_create_sync(C.byref(h)), "event_create_sync")
                return h
            self._evs = {"fork_pool": [mk(), mk()], "pooled": [mk(), mk()], "fork": mk(), "join": mk()}
        return self._evs

    @_on_device
    def x_past(self):
        """[Bv, e, S+L] ([Bv, e, L] after a first chunk): what the reference keeps as `x_past` (gibbs:215,221) -- the
        re-sampled rows of the previous coefficients followed by the pooled frames of the most recent call."""
        if self._last_ragged:
            raise RuntimeError("x_past: the last call was a ragged step (per-video lengths); its pooled frames are not "
                               "kept -- x_past is defined for lock-step calls only")
        xp = self._last_xpart
        if xp is None:                      # the last call pooled per bin: pool the chunk again, per frame
            k = self._last_k() if getattr(self, "_last_k", None) is not None else None
            if k is None:
                raise RuntimeError("x_past: the frames of the last chunk were pooled per bin and the chunk tensor is "
                                   "gone; construct the engine with bin_pool=False to keep them")
            xp = self.pool(k)
        x = xp.sum(2) if xp.shape[2] > 1 else xp[:, :, 0]                                              # [Bv,L,e]
        if not self._last_updated:
            return x.transpose(1, 2)
        idx = self.last["idx"] if self.sticky else \
            tables.rect_tables(self._last_L, self.N, self.tau, self.S, spacing=self.spacing).to(self.device)[
                "idx_uniform"].unsqueeze(0).expand(x.shape[0], -1).contiguous()
        xm = ops.gather_rows(self._B[1 - self._cur], idx)                   # previous coefficients: other buffer
        return torch.cat([xm, x], 1).transpose(1, 2)

    @_on_device
    def density(self):
        """alphas[Q,Bv,H,768] of the most recent call: the density side-output the Video-LLaMA copy pickles to
        ./alphas_uniform on every forward (gibbs:320-343).  Needs `keep_scores=True`."""
        sc = self.last.get("scores")
        if sc is None:
            raise RuntimeError("density() needs the scores of the last call: construct with keep_scores=True")
        L = self._last_L
        td = tables.rect_tables(L, self.N, self.tau, self.S, spacing=self.spacing).to(self.device)
        return ops.density_rect(sc, td["jd"], td["wd"])

    @_on_device
    def pool(self, k, with_half=False, lengths=None, chunk_frames=None):
        """Frame pooling alone (gibbs:304): k[Bv, L*T, e] -> pooled frames [Bv, L, splits, e].  The result can be
        handed to `step(..., pooled=...)` of SEVERAL engines: every LTM layer of a Q-former receives the same
        `encoder_hidden_states` per chunk (2 layers in Video-LLaMA, 6 in VideoChat2; SURVEY section 8f N2), so the
        25 MB/video chunk needs to be streamed from HBM once, not once per layer.
        `with_half=True` (fp32 chunks): the same pass also writes the chunk as float16 and returns
        (pooled, k16[Bv, L*T, e]) -- the operand of the caller's short-term attention (SURVEY 8f N1).
        `lengths` (ragged chunk, see `step`): only the first lengths[v] frames of video v are pooled and read; the
        result is packed video after video, [sum(lengths), splits, e] with splits = `_splits(sum(lengths))`, and is
        handed to `step(..., pooled=..., lengths=...)` with the same lengths.  With `with_half` (fp32 chunks) it comes
        with k16[Bv, ld16, e], ld16 = L*T rounded up to 64 tokens: video v's first n_v = lengths[v]*T tokens as fp16,
        zeros up to roundup64(n_v), the rest unwritten (ltm_pool_mean_convert_ragged).
        `k` may be a list of per-video entries with `chunk_frames` (see `step`): the packed frames as for `lengths`,
        read from each entry where it lives (no `with_half`)."""
        k = self._entries(k, chunk_frames, lengths)
        if isinstance(k, _Entries):
            if with_half:
                raise ValueError("with_half: a chunk given as a list is pooled without the fp16 copy")
            Bv, LT, e = k.shape
            frames = sum(k.lens)
            splits = self._splits(frames)
            out = torch.empty(frames, splits, e, device=self.device, dtype=torch.float32)
            if frames:
                _, offs, table = self._lengths_dev(k.lens, k.ptrs)
                ops.pool_ptrs(table, k.code, out, offs, Bv, LT // self.T, self.T, e, splits, frames)
            return out
        require_cuda(k)
        k = k.contiguous()
        Bv, LT, e = k.shape
        if e != self.e or LT % self.T:
            raise ValueError(f"k must be [Bv, L*{self.T}, {self.e}]")
        L = LT // self.T
        if lengths is not None:
            if k.dtype not in ops.CHUNK_DTYPES or (with_half and k.dtype != torch.float32):
                raise ValueError("a ragged chunk is pooled from float32 / float16 / bfloat16 storage (with_half: float32)")
            lens = _as_lengths(lengths, Bv, L)
            frames = sum(lens)
            splits = self._splits(frames)
            if with_half:
                return ops.pool_mean_convert_ragged(k.view(Bv, L, self.T, e), self._lengths_dev(lens)[1], frames, splits,
                                                    (LT + 63) // 64 * 64)
            out = torch.empty(frames, splits, e, device=self.device, dtype=torch.float32)
            if frames:
                ops.pool_into(k, out, L, self.T, splits, offs=self._lengths_dev(lens)[1], frames=frames)
            return out
        if with_half:
            x, k16 = ops.pool_mean_convert(k.view(Bv, L, self.T, e), self._splits(Bv * L))
            return x, k16.view(Bv, LT, e)
        return ops.pool_mean(k.view(Bv, L, self.T, e), self._splits(Bv * L))

    @_on_device
    def step(self, k, q, u=None, new_doc=False, pooled=None, beside_pooling=False, lengths=None, chunk_frames=None):
        """k[Bv, L*T, e] float32 / float16 / bfloat16 (16-bit: e % 8 == 0, pooled per frame from its own storage),
        q[Bv,Q,D] float32, CUDA; u[Bv,S] fp64 uniforms (needed from the second chunk on when
        sticky); new_doc: bool or per-video flags; pooled: result of `pool(k)` (then `k` is only used for its
        shape); beside_pooling: the caller pools another chunk on a second stream while this step runs (the K/V
        projection then keeps to part of the SMs, see `gemm_ctas_overlap`).  Returns ctx[Bv,Q,D].

        lengths (ragged batch): Bv host integers, each 0 or in [2, L].  Video v uses the first lengths[v] frames of
        its padded chunk (the rest is never read and may hold anything); lengths[v] == 0 leaves video v idle: its
        memory is kept bit for bit, its row of u is not read and its ctx rows are zero (with new_doc[v] the slot is
        cleared instead).  new_doc is then a bool or host flags; a slot without memory must receive new_doc with its
        first chunk.  Passing lengths always takes the ragged kernels, even when all lengths are equal.

        k as a list (per-video chunks, no padded copy): Bv entries, each None (the slot is idle, length 0) or a CUDA
        tensor [n_v*T, e] with 2 <= n_v <= chunk_frames, dense rows (strides (e, 1)) and a 16-byte aligned start --
        separate tensors, chunk views of whole-video tensors (`video.split_videos`) or views into one packed tensor.
        The present entries share one dtype (float32 / float16 / bfloat16).  chunk_frames (required) is the padded
        length L that selects the tables and workspace; the lengths follow from the entries (passing `lengths` too is
        a ValueError).  Everything else is the ragged step above, bit for bit: each frame is pooled where it lives."""
        k = self._entries(k, chunk_frames, lengths)
        lst = isinstance(k, _Entries)
        require_cuda(q, u, None if lst else k)
        kdt = (k.code if lst else self._chunk_dtype(k)) if pooled is None else 0   # (with `pooled`, k gives the shape)
        if q.dtype != torch.float32:
            raise ValueError("q must be float32")
        k, q = (k if lst else k.contiguous()), q.contiguous()
        Bv, L, Q, tab, tdev, flags, u, rag = self._prepare(k, q, new_doc, u, k.lens if lst else lengths, pooled,
                                                           ptrs=k.ptrs if lst else None)
        ws = self._workspace(Bv, L, Q)
        if rag is not None:
            self._ragged_ws(ws, Bv, L)
        ctx = torch.empty(Bv, Q, self.D, device=self.device, dtype=torch.float32)
        hit = self._frames_source(k, Q, ws, tab, flags, rag, pooled)
        main = torch.cuda.current_stream(self.device)
        run = main
        if hit is not None:
            run = self._compute                      # fork: high-priority compute stream, joined below
            ev = self._sync_events()
            rp, mp = C.c_void_p(run.cuda_stream), C.c_void_p(main.cuda_stream)
            check(lib().ltm_event_record(ev["fork"], mp), "event_record")
            check(lib().ltm_stream_wait_event(rp, ev["fork"]), "stream_wait_event")
            # (a graph capture cannot wait on an event recorded before it began: the capturing host has synchronised,
            # and on replay the buffer is the one the previous replay's last prefetch filled)
            if hit["captured"] or not torch.cuda.is_current_stream_capturing():
                check(lib().ltm_stream_wait_event(rp, hit["event"]), "stream_wait_event")
        # (a pending prefetch = the next chunk is being pooled on the side stream while this step runs)
        beside = bool(beside_pooling) or (pooled is None and bool(self._pref))
        a = self._args(Bv, L, Q, ws, tab, tdev, beside_pool=beside, rag=rag, k_dtype=kdt)
        if pooled is not None:
            a.xpart, a.splits, a.binned = pooled.data_ptr(), pooled.shape[-2], 0
        if rag is not None and run is not main:
            rag["lens_dev"].record_stream(run)
        pool_here = pooled is None and hit is None
        if pool_here and lst:
            a.k_ptrs = rag["ptrs_dev"].data_ptr()
        check(lib().ltm_rect_step(C.byref(a), ptr(k) if pool_here and not lst else None, ptr(q), ptr(u), ptr(flags),
                                  ptr(ctx), C.c_void_p(run.cuda_stream)), "rect_step")
        if hit is not None:
            check(lib().ltm_event_record(ev["join"], rp), "event_record")
            check(lib().ltm_stream_wait_event(mp, ev["join"]), "stream_wait_event")
        self._finish(ws, pooled, k=k, rag=rag)
        return ctx

    @_on_device
    def step_overlapped(self, k, q, u=None, new_doc=False, k_next=None, next_new_doc=False, lengths=None,
                        next_lengths=None, chunk_frames=None):
        """`step(k, ...)` with the frame pooling of `k_next` issued beside it, in ONE library call
        (`ltm_rect_step_overlap`: side stream pools the next chunk, a high-priority stream runs this chunk's
        regression / projection / attention, the current stream joins both).  `k` must be the tensor handed over as
        `k_next` by the previous call (or to `prefetch`); the first chunk of a stream is pooled here.  Same results as
        `step`, bit for bit.  `next_new_doc=True` says that `k_next` will start new documents (then it is pooled per
        frame; a chunk expected to continue the videos may be pooled per bin, see `bin_pool`).
        `lengths` / `next_lengths`: per-video lengths of `k` / `k_next` (ragged chunks, see `step`); `k` is matched
        with its prefetch by lengths too.  `k` and `k_next` are float32, float16 or bfloat16, each on its own (see
        `step`); `q` is float32.  `k` and `k_next` may each be a list of per-video entries (see `step`), with
        `chunk_frames` = L; a padded `k` or `k_next` then has L*T tokens."""
        listed = [isinstance(x, (list, tuple)) for x in (k, k_next)]
        if chunk_frames is not None and not any(listed):
            raise ValueError("chunk_frames applies to a chunk given as a list")
        k = self._entries(k, chunk_frames if listed[0] else None, lengths)
        k_next = self._entries(k_next, chunk_frames if listed[1] else None, next_lengths, "k_next")
        lst, nlst = isinstance(k, _Entries), isinstance(k_next, _Entries)
        require_cuda(q, u, None if lst else k, None if (nlst or k_next is None) else k_next)
        kdt = k.code if lst else self._chunk_dtype(k)
        ndt = 0 if k_next is None else k_next.code if nlst else self._chunk_dtype(k_next, "k_next")
        if q.dtype != torch.float32:
            raise ValueError("q must be float32")
        if chunk_frames is not None and k.shape[1] != int(chunk_frames) * self.T:
            raise ValueError(f"k has {k.shape[1]} tokens, chunk_frames={chunk_frames} means {int(chunk_frames) * self.T}")
        if k_next is not None and ((not nlst and not k_next.is_contiguous()) or tuple(k_next.shape) != tuple(k.shape)):
            raise ValueError("k_next must be contiguous and have the shape of k (a list: as many entries as k has "
                             "videos)")
        nl = None
        if nlst:
            nl = k_next.lens
        elif k_next is not None and next_lengths is not None:
            nl = _as_lengths(next_lengths, k.shape[0], k.shape[1] // self.T)
        k, q = (k if lst else k.contiguous()), q.contiguous()
        Bv, L, Q, tab, tdev, flags, u, rag = self._prepare(k, q, new_doc, u, k.lens if lst else lengths)
        ws = self._workspace(Bv, L, Q)
        if rag is not None or nl is not None:
            self._ragged_ws(ws, Bv, L)
        hit = self._frames_source(k, Q, ws, tab, flags, rag, prefetch=True)
        ev = self._sync_events()
        main = torch.cuda.current_stream(self.device)
        capturing = torch.cuda.is_current_stream_capturing()
        o = Overlap()
        o.main_stream, o.side_stream, o.compute_stream = main.cuda_stream, self._side.cuda_stream, self._compute.cuda_stream
        o.ev_fork, o.ev_join = ev["fork"], ev["join"]
        o.ev_pooled_cur = hit["event"] if (hit["captured"] or not capturing) else None
        o.pool_ctas = int(self.pool_ctas)
        if k_next is not None:
            b = self._pref_buffer(ws)
            if nl is not None:
                nl_dev, noffs_dev, ntab = self._lengths_dev(nl, k_next.ptrs if nlst else None)
                nl_dev.record_stream(self._side)        # (with the table: one buffer)
                nf = sum(nl)
                o.next_lengths, o.next_offs = nl_dev.data_ptr(), noffs_dev.data_ptr()
                o.next_frames, o.next_splits = nf, self._splits(nf)
                o.next_ptrs = ntab.data_ptr() if nlst else None
                nb = False
            else:
                nb = (not next_new_doc) and self._bin_ok(Bv, L, tab, ndt)
            o.k_next = None if nlst else k_next.data_ptr()
            o.xpart_next, o.next_binned = ws["xbufs"][b].data_ptr(), int(nb)
            o.next_dtype = ndt
            o.ev_fork_pool, o.ev_pooled_next = ev["fork_pool"][b], ev["pooled"][b]
            for t in (k_next.stores if nlst else (k_next,)):
                t.record_stream(self._side)
            self._pref.append(dict(refs=_chunk_refs(k_next), buf=b, event=ev["pooled"][b], captured=capturing,
                                   binned=nb, lens=nl))
        ctx = torch.empty(Bv, Q, self.D, device=self.device, dtype=torch.float32)   # main joins the compute stream
        a = self._args(Bv, L, Q, ws, tab, tdev, beside_pool=k_next is not None, rag=rag, k_dtype=kdt)
        if rag is not None:
            rag["lens_dev"].record_stream(self._compute)
        check(lib().ltm_rect_step_overlap(C.byref(a), C.byref(o), ptr(q), ptr(u), ptr(flags), ptr(ctx)),
              "rect_step_overlap")
        self._finish(ws, k=k, rag=rag)
        return ctx

    @_on_device
    def step_host(self, k_host, q_host, u_host=None, new_doc=False, out=None):
        """Same as `step` but through HOST buffers (ideally pinned): the C entry point enqueues the H2D copies,
        the kernels and the D2H copy of ctx on the current stream.  Returns the host ctx tensor; the caller
        synchronises the stream before reading it.  k_host is float32, float16 or bfloat16 (a 16-bit chunk is copied
        as it is: half the H2D bytes); q_host float32."""
        if k_host.is_cuda or q_host.is_cuda:
            raise ValueError("step_host takes host tensors")
        kdt = self._chunk_dtype(k_host, "k_host")
        if q_host.dtype != torch.float32:
            raise ValueError("step_host takes float32 q")
        Bv, L, Q, tab, tdev, flags, u_host, _ = self._prepare(k_host, q_host, new_doc, u_host, u_name="u_host")
        ws = self._workspace(Bv, L, Q)
        dev = self.device
        if ws["k_dev"] is None or ws["k_dev"].dtype != k_host.dtype:
            # staging buffer in the chunk's own storage: the H2D copy moves 2 bytes per element for a 16-bit chunk
            ws["k_dev"] = torch.empty(Bv, L * self.T, self.e, device=dev, dtype=k_host.dtype)
        if ws["q_dev"] is None:
            ws["q_dev"] = torch.empty(Bv, Q, self.D, device=dev, dtype=torch.float32)
            ws["u_dev"] = torch.empty(Bv, self.S, device=dev, dtype=torch.float64)
            ws["nd_dev"] = torch.empty(Bv, device=dev, dtype=torch.uint8)
            ws["ctx_dev"] = torch.empty(Bv, Q, self.D, device=dev, dtype=torch.float32)
        if out is None:
            out = torch.empty(Bv, Q, self.D, dtype=torch.float32, pin_memory=True)
        ws["xtag"][ws["xi"]] = False          # the host path pools per frame
        a = self._args(Bv, L, Q, ws, tab, tdev, k_dtype=kdt)
        a.k_dev = ws["k_dev"].data_ptr()      # (the cached block may hold a staging buffer of another dtype)
        nd_host = None
        if flags is not None:
            nd_host = torch.as_tensor(new_doc).to(torch.uint8).contiguous()
        check(lib().ltm_rect_step_host(C.byref(a), ptr(k_host.contiguous()), ptr(q_host.contiguous()), ptr(u_host),
                                       ptr(nd_host), ptr(out), stream_ptr(dev)), "rect_step_host")
        self._keep = (k_host, q_host, u_host, nd_host)      # keep host buffers alive until the stream drains
        self._finish(ws)
        return out


class BatchedGaussLTM(_BatchedBase):
    """Variant G: Gaussian RBF bases, dense ridge regression, closed-form continuous softmax
    (long_term_attention.py:259-325).  `k` is consumed un-pooled: [Bv, Lk, e]."""

    def __init__(self, num_basis, tau, w_key, b_key, w_value, b_value, *, sigmas=(0.005, 0.01), n_heads=12,
                 head_size=64, sticky=True, nb_samples=tables.NB_SAMPLES, precision="tf32x3",
                 proj_precision=None, device="cuda", ridge=tables.RIDGE_PENALTY,
                 spacing="linear", value_precision=None, fold_samples=True, tc_attn=True):
        ns = len(sigmas)
        n = int(num_basis)
        if n % ns:
            n += ns - n % ns
        super().__init__(n, tau, w_key, b_key, w_value, b_value, n_heads, head_size, sticky, nb_samples,
                         precision, device)
        self.sigmas = tuple(float(s) for s in sigmas)
        self.spacing = spacing
        # K/V projection (three quarters of the variant's flops): "fp16x2" (default) = operands split into two fp16 terms
        # each (22 significant bits) and laid out along K so that ONE plain kind::f16 GEMM over 3e computes the
        # three-term product (ops.split_half3): as accurate as split-TF32 (4e-6 vs 6e-6 against fp64) at the fp16
        # tensor rate, 370 -> 202 + 39 us per 128-video chunk.  fp16's range applies to the coefficients (|B| <= 65504);
        # "tf32x3" keeps the fp32 operands.
        self.proj_precision = proj_precision or ("fp16x2" if precision == "tf32x3" else precision)
        # precision of the value half of the projection: None (default) = split-TF32 like the keys.  Both cheaper
        # options were measured and miss the 1e-3 context tolerance: "tf32" (single pass on the fp32 operands; the
        # tensor core TRUNCATES them, a systematic ~1e-3 shrink of V; 128.7 k -> 161.3 k chunks/s) and "fp16" (operands
        # rounded to fp16 first: unbiased, but the Gaussian weights r_j reach ~80 with mixed signs downstream of the
        # ridge operators and amplify the 2^-12 rounding to 1.15e-3; 143 k -> 161.8 k).
        self.value_precision = value_precision
        # sticky update as A_v [R ; k] with the operator's sample columns folded per drawn bin (ltm_fold_sample_columns)
        # instead of G_inf^T [gather(R) ; k]: same B, no [Bv,S,e] intermediate, contraction 128 + L instead of S + L
        self.fold_samples = bool(fold_samples)
        self._W3 = None
        # tensor-core attention (csrc/attn_g16.cu): num_basis 64 / 128 / 256, head size 64, with the fp16x2 projection
        self.tc_attn = (bool(tc_attn) and self.proj_precision == "fp16x2" and ops.attn_tc_supported(self.N, self.d)
                        and self.value_precision is None and self.e % 8 == 0)
        self.ridge = float(ridge)
        self._ops = {}
        self._B = None
        self.last = {}

    # ------------------------------------------------------------------ constant operators
    @_on_device
    def operators(self, L):
        """Device tables + ridge operators for chunk length L (solved once, fp64, on the device)."""
        op = self._ops.get((L, self.spacing))
        if op is None:
            t = tables.gauss_tables(L, self.N, self.tau, self.sigmas, self.S, spacing=self.spacing)
            dev = self.device
            f = lambda a: torch.from_numpy(a).to(dev)
            op = dict(t=t, mu=f(t.basis_mu), sigma=f(t.basis_sigma), tb=f(t.tb), bins=f(t.bins))
            _, op["G0T"] = ops.ridge_solve(f(t.pos0), t.trim0, L, op["mu"], op["sigma"], self.ridge,
                                           want_G=False, want_GT=True)                       # [N, L]
            _, op["GinfT"] = ops.ridge_solve(f(t.pos1), t.trim1, self.S + L, op["mu"], op["sigma"], self.ridge,
                                             want_G=False, want_GT=True)                     # [N, S+L]
            # design of the 128 possible sticky sample positions (bins[b], b=0..127): rows of Psi
            op["Psi_tab"] = ops.rbf_eval(op["bins"][:128].contiguous(), op["mu"], op["sigma"])   # [128, N]
            op["Psi_uniform"] = ops.rbf_eval(f(t.old_over_tau), op["mu"], op["sigma"])           # [S, N]
            self._ops[(L, self.spacing)] = op
        return op

    @_on_device
    def set_operators(self, L, G0=None, G_inf=None):
        """Inject ridge operators ([L,N] / [S+L,N]) computed elsewhere (used by the parity tests to share
        the reference's fp32 `.inverse()` result, see DESIGN.md)."""
        op = self.operators(L)
        if G0 is not None:
            op["G0T"] = _pad_rows(G0.to(self.device, torch.float32).t())
        if G_inf is not None:
            op["GinfT"] = _pad_rows(G_inf.to(self.device, torch.float32).t())

    @property
    def B_past(self):
        return self._B if self.has_state else None

    @_on_device
    def step(self, k, q, u=None, new_doc=False):
        """k[Bv,Lk,e], q[Bv,Q,D], u[Bv,S] fp64.  Returns ctx[Bv,Q,D]."""
        require_cuda(k, q, u)
        if k.dtype != torch.float32 or q.dtype != torch.float32:
            raise ValueError("k and q must be float32")
        k, q = k.contiguous(), q.contiguous()
        Bv, L, e = k.shape
        if e != self.e:
            raise ValueError(f"k has width {e}, projections expect {self.e}")
        if self.Bv != Bv:
            self.Bv, self.has_state = Bv, False
        if not isinstance(new_doc, (bool, int)):
            return self._step_mixed(k, q, u, new_doc)
        if new_doc:
            self.has_state = False
        op = self.operators(L)
        info = {}
        if not self.has_state:
            # B = G0^T k      (A = G0T [N,L] K-major, shared;  B = k[v] [L,e] MN-major)
            B = ops.gemm(op["G0T"], k, a_kmajor=True, b_kmajor=False, precision=self.precision, impl=self.gemm_impl)
        else:
            if self.sticky:
                if u is None or u.dtype != torch.float64 or tuple(u.shape) != (Bv, self.S):
                    raise ValueError(f"sticky re-sampling needs u: float64 [{Bv},{self.S}]")
                hist = ops.sticky_hist_gauss(self._mu, self._sd, op["tb"])
                rs = ops.resample(hist, u.contiguous(), op["bins"], None, normalize=True, sort=True)
                info.update(p=rs["p"], b=rs["b_draw"], b_sorted=rs["b_used"], ts=rs["ts"])
                # reconstruct the old signal at the 128 candidate positions, then gather the 512 drawn rows:
                # xm[s] = Psi(ts_s) B_past  ==  (Psi_tab B_past)[b_s]
                R = ops.gemm(op["Psi_tab"], self._B, a_kmajor=True, b_kmajor=False, precision=self.precision,
                             impl=self.gemm_impl)                                          # [Bv,128,e]
                if self.fold_samples:
                    # G_inf^T [xm ; k] = A_v [R ; k]: the sample columns of the operator summed per drawn bin (the
                    # draws are sorted), so the 512 gathered rows are never written and the contraction is 128 + L long
                    A_v = ops.fold_sample_columns(op["GinfT"], rs["b_used"], self.S, L)     # [Bv,N,128+L]
                    B = ops.gemm(A_v, R, B2=k, a_kmajor=True, b_kmajor=False, precision=self.precision,
                                 impl=self.gemm_impl)
                    xm = None
                else:
                    xm = ops.gather_rows(R, rs["b_used"])                                   # [Bv,S,e]
            else:
                xm = ops.gemm(op["Psi_uniform"], self._B, a_kmajor=True, b_kmajor=False, precision=self.precision,
                              impl=self.gemm_impl)
            if xm is not None:
                # B = G_inf^T [xm ; k]  without materialising the concatenation
                B = ops.gemm(op["GinfT"], xm, B2=k, a_kmajor=True, b_kmajor=False, precision=self.precision,
                             impl=self.gemm_impl)
        self._B = B
        if self.tc_attn:
            # tensor-core path: K|V straight out of the fp16x2 projection as two fp16 terms, both attention
            # contractions as kind::f16 UMMAs over the two-term operands (csrc/attn_g16.cu)
            if self._W3 is None or self._W3_src != self.Wkv.data_ptr():
                self._W3, self._W3_src = ops.split_half3(self.Wkv, 1), self.Wkv.data_ptr()
            KVh, KVl = ops.project_kv_split(B, self.bkv, self.N, self._W3)
            ctx, mu, sd = ops.cont_attn_gauss_tc16(q, KVh, KVl, op["mu"], op["sigma"], n_heads=self.H)
        elif ops.attn_fast_supported(self.N, self.d):
            w3 = None
            if self.proj_precision == "fp16x2":
                if self._W3 is None or self._W3_src != self.Wkv.data_ptr():
                    self._W3, self._W3_src = ops.split_half3(self.Wkv, 1), self.Wkv.data_ptr()
                w3 = self._W3
            Kt, V = ops.project_kv_t(B, self.Wkv, self.bkv, self.N, precision=self.proj_precision,
                                     impl=self.gemm_impl, precision_v=self.value_precision, w_split=w3)
            ctx, scores, mu, sd = ops.cont_attn_gauss_t(q, Kt, V, op["mu"], op["sigma"])
        else:
            pp = self.precision if self.proj_precision == "fp16x2" else self.proj_precision      # (generic layout: fp32 operands)
            KV = ops.project_kv(B, self.Wkv, self.bkv, precision=pp, impl=self.gemm_impl)
            KV = KV.view(Bv, self.N, 2 * self.D)
            ctx, scores, mu, sd = ops.cont_attn_gauss(q, KV, op["mu"], op["sigma"], n_heads=self.H)
        self._mu, self._sd = mu, sd
        self.has_state = True
        info.update(mu=mu, sd=sd)
        self.last = info
        return ctx


def _gauss_step_mixed(self, k, q, u, new_doc):
    """Per-video new_doc flags (host booleans): the videos that start a new document and those that continue run
    through the two branches as two sub-batches; the per-video state is split and merged around them."""
    flags = torch.as_tensor(new_doc).to("cpu", torch.bool).reshape(-1)
    Bv = k.shape[0]
    if flags.numel() != Bv:
        raise ValueError("new_doc must be a bool or one flag per video")
    if not self.has_state or bool(flags.all()):
        return self.step(k, q, u, new_doc=True)
    if not bool(flags.any()):
        return self.step(k, q, u, new_doc=False)
    dev = self.device
    fi = flags.nonzero().flatten().to(dev)
    ci = (~flags).nonzero().flatten().to(dev)
    state = (self._B, self._mu, self._sd)
    ctx = torch.empty(Bv, q.shape[1], self.D, device=dev, dtype=torch.float32)
    outs = {}
    for sel, first in ((ci, False), (fi, True)):
        self.Bv = int(sel.numel())
        self.has_state = not first
        if not first:
            self._B, self._mu, self._sd = state[0][sel].contiguous(), state[1][sel].contiguous(), state[2][sel].contiguous()
        ctx[sel] = self.step(k[sel].contiguous(), q[sel].contiguous(), None if (first or u is None) else u[sel].contiguous(),
                             new_doc=first)
        outs[first] = (self._B, self._mu, self._sd)
    B = torch.empty_like(state[0]); mu = torch.empty_like(state[1]); sd = torch.empty_like(state[2])
    for sel, first in ((ci, False), (fi, True)):
        B[sel], mu[sel], sd[sel] = outs[first]
    self._B, self._mu, self._sd = B, mu, sd
    self.Bv, self.has_state = Bv, True
    self.last = dict(mu=mu, sd=sd)
    return ctx


def _gauss_kl(self, mu_0, sigma_0):
    """KL regulariser of the most recent call, [Bv, H*Q] (long_term_attention.py:296-304)."""
    return ops.kl_gauss(self._mu, self._sd, mu_0, sigma_0)


def _gauss_x_past(self):
    return None


BatchedGaussLTM._step_mixed = _gauss_step_mixed
BatchedGaussLTM.kl = _on_device(_gauss_kl)
BatchedGaussLTM.x_past = _gauss_x_past


def BatchedLTM(variant="gibbs", **kw):
    """Factory: variant in {"gibbs", "gaussian"}."""
    if variant in ("gibbs", "rect", "R"):
        return BatchedRectLTM(**kw)
    if variant in ("gaussian", "gauss", "G"):
        return BatchedGaussLTM(**kw)
    raise ValueError(f"unknown LTM variant {variant!r}")
