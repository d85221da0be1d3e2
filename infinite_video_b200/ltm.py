"""Drop-in `LongTermAttention` for the infinity-Video Q-formers, executing on libinfltm (sm_100a).

Mirrors the constructor and `forward(k, q, new_doc, layer_n)` of the reference module
(infty-Video-LLaMA/InfVideoLLaMA/models/long_term_attention_gibbs.py:25-65,288-346 -- the live
"gibbs" variant imported by Qformer.py:50 -- and .../long_term_attention.py:25-67,259-392 for the
Gaussian variant).  The caller (`BertSelfAttention`, Qformer.py:135-158,216-223) constructs it through a
keyword `partial`, writes `.length` / `.target_len` before each call, passes its own `key` / `value`
`nn.Linear` modules as `proj_key` / `proj_value`, and `.detach()`es the result.

Install by swapping one import (Qformer.py:50):
    from infinite_video_b200 import LongTermAttention

Differences that are deliberate (DESIGN.md section "boundary"):
  * constant tables are cached per (L, N, tau) instead of being rebuilt on the CPU every call;
  * the uniform draws of the sticky re-sampling are explicit: `u=` (float64 [B,512]) or a
    `torch.Generator`; by default they are taken from torch's global CPU generator in the same
    amount and order as the reference running on CPU (512 used + 512 discarded fp64 draws per call);
  * a batch of B > 1 independent videos is accepted (the reference hard-wires B = 1);
  * the Video-LLaMA copy's per-call pickle of the attention density to ./alphas_uniform
    (gibbs:320-345) is not written.
"""
import weakref

import numpy as np
import torch
import torch.nn as nn

from . import tables
from .batched import BatchedGaussLTM, BatchedRectLTM, _as_lengths


class LongTermAttention(nn.Module):
    # Pooled frames of the most recent chunk, shared by every instance in the process: all LTM layers of a
    # Q-former are called with the same `encoder_hidden_states` tensor per chunk (Qformer.py:216-223 inside
    # BertEncoder's layer loop), so only the first layer streams the chunk from HBM (SURVEY section 8f N2).
    _shared_pool = {"key": None, "x": None, "k16": None}

    def __init__(self, head_size: int, length: int, target_len: int, attn_func: str, attn_num_basis: int,
                 continuous: bool, attn_drop: float, infinite_memory: bool, n_layers: int, n_heads: int,
                 affines: bool, mask: bool, mask_type: str, kl_regularizer: bool, proj_key, proj_value,
                 sigma_0, mu_0, sticky_memories, sigmas, tau, variant: str = "gibbs",
                 tokens_per_frame: int = 32, precision: str = None,
                 share_pooling: bool = True, output_density: bool = False, dump_path: str = None,
                 kv_dtype: str = "fp16", **kwargs):
        super().__init__()
        if not continuous:
            raise NotImplementedError("only the continuous-attention memory is on the LTM path (continuous=True)")
        if not infinite_memory:
            raise NotImplementedError("infinite_memory=False is never used by the Q-formers (Qformer.py:141)")
        if attn_func != "softmax":
            raise NotImplementedError("attn_func must be 'softmax' (Qformer.py:140)")
        if variant not in ("gibbs", "gaussian"):
            raise ValueError("variant must be 'gibbs' (live module) or 'gaussian'")
        if kl_regularizer and variant != "gaussian":
            raise NotImplementedError("kl_regularizer exists in the Gaussian variant only (long_term_attention.py:296-304)")
        if kl_regularizer and (sigma_0 is None or mu_0 is None):
            raise ValueError("kl_regularizer needs sigma_0 and mu_0")
        # same attribute surface as the reference (gibbs:32-65)
        self.device = "cuda"
        self.length = length
        self.target_len = target_len
        self.head_size = head_size
        self.attn_num_basis = attn_num_basis
        self.continuous = continuous
        self.attn_func = attn_func
        self.n_head = n_heads
        self.sigmas = sigmas
        self.kl_regularizer = kl_regularizer
        self.sigma_0 = sigma_0
        self.mu_0 = mu_0
        # the caller's nn.Linear modules; not registered as sub-modules twice on purpose: the reference
        # stores them as plain attributes of an nn.Module as well (which registers them) -> keep parity
        self.proj_key = proj_key
        self.proj_value = proj_value
        self.affines = affines
        self.sticky_memories = sticky_memories
        self.mem_threshold = 2048
        self.infinite_memory = infinite_memory
        self.nb_samples = tables.NB_SAMPLES
        self.tau = tau
        self.count = 0
        self.ridge_penalty = tables.RIDGE_PENALTY
        self.padding = True
        self.spacing = "linear"
        self.variant = variant
        self.tokens_per_frame = tokens_per_frame
        self.precision = precision
        self.share_pooling = share_pooling
        # storage of the projected keys / values between calls: "fp16" (default; same 11-bit significand as the tf32
        # grid, half the bytes, |K|,|V| <= 65504) or "fp32"
        self.kv_dtype = kv_dtype
        # Video-LLaMA copy: density side-output of every call (gibbs:320-343).  Off by default; when on, the
        # result is kept on the device in `self.alphas` ([Q,B,H,768]) instead of being pickled to the cwd.
        # `dump_path` (e.g. "./alphas_uniform", what the Video-LLaMA copy hard-codes at gibbs:344-345): additionally
        # pickle the CPU copy of that tensor on every call, the file relevant_frames.py:11-12 reads.
        self.output_density = bool(output_density) or dump_path is not None
        self.dump_path = dump_path
        self.alphas = None
        self.kl_reg = None
        self._engine = None
        self._wver = None

    # ------------------------------------------------------------------ engine / weights
    def _weights_version(self):
        ps = [self.proj_key.weight, self.proj_key.bias, self.proj_value.weight, self.proj_value.bias]
        return tuple((p.data_ptr(), p._version) if p is not None else None for p in ps)

    def _get_engine(self, device):
        ver = self._weights_version()
        if self._engine is None or self._engine.device != device:
            common = dict(num_basis=self.attn_num_basis, tau=self.tau, w_key=self.proj_key.weight,
                          b_key=self.proj_key.bias, w_value=self.proj_value.weight, b_value=self.proj_value.bias,
                          n_heads=self.n_head, head_size=self.head_size, sticky=bool(self.sticky_memories),
                          nb_samples=self.nb_samples, device=device)
            if self.variant == "gibbs":
                self._engine = BatchedRectLTM(tokens_per_frame=self.tokens_per_frame,
                                              precision=self.precision or "tf32",
                                              keep_scores=self.output_density, spacing=self.spacing,
                                              kv_dtype=self.kv_dtype, **common)
            else:
                sig = self.sigmas if self.sigmas is not None else (0.005, 0.01)
                self._engine = BatchedGaussLTM(sigmas=tuple(sig), precision=self.precision or "tf32x3",
                                               spacing=self.spacing, **common)
            self._wver = ver
        elif ver != self._wver:
            self._engine.set_projections(self.proj_key.weight, self.proj_key.bias, self.proj_value.weight,
                                         self.proj_value.bias)
            self._wver = ver
        if self._engine.spacing != self.spacing:        # plain attribute upstream (gibbs:64): honoured when changed
            self._engine.spacing = self.spacing
            self._engine.reset()
        return self._engine

    @property
    def x_past(self):
        """[B, e, S+L] regression input of the most recent call, as the reference keeps it (gibbs:221): the 512
        contracted re-samples of the old memory followed by the pooled frames ([B, e, L] after a first chunk).
        Assembled on demand; None before the first call and for the Gaussian variant fed with 16-bit chunks."""
        eng = self._engine
        return None if eng is None or not eng.has_state else eng.x_past()

    @x_past.setter
    def x_past(self, value):
        if value is not None:
            raise AttributeError("x_past can only be cleared (set to None)")

    @property
    def B_past(self):
        return None if self._engine is None else self._engine.B_past

    @B_past.setter
    def B_past(self, value):
        if value is not None:
            raise AttributeError("B_past can only be cleared (set to None)")
        if self._engine is not None:
            self._engine.reset()

    # ------------------------------------------------------------------ forward
    def _draw_uniforms(self, bsz, generator):
        # Categorical(p).sample((512,)) consumes bsz*512 fp64 draws, the dummy bins_cat.sample((512, 1))
        # another 512 that are thrown away (gibbs:205-206; SURVEY.md A11).
        u = torch.rand(bsz, self.nb_samples, dtype=torch.float64, generator=generator)
        torch.rand(self.nb_samples, dtype=torch.float64, generator=generator)
        return u

    def check_ragged(self, k, lengths, new_doc, Q):
        """Host-side validation of a ragged call with Q queries per video, before anything is launched: lengths (host
        ints, each 0 or in [2, L]), new_doc (a bool or one host flag per video), that every present video that does not
        start a new document has memory to continue, and that no video holding memory sees its number of query tiles
        change without new_doc (the checks `BatchedRectLTM.step` makes).  Returns (lengths tuple, bool ndarray of
        new_doc flags)."""
        if self.variant != "gibbs":
            raise NotImplementedError("per-video lengths exist for variant 'gibbs' only")
        bsz, LT = k.shape[0], k.shape[1]
        if LT % self.tokens_per_frame or LT // self.tokens_per_frame < 2:
            raise ValueError(f"k has {LT} tokens: a ragged chunk is padded to L*{self.tokens_per_frame} tokens, L >= 2")
        lens = _as_lengths(lengths, bsz, LT // self.tokens_per_frame)
        if isinstance(new_doc, (bool, int)):
            nd = np.full(bsz, bool(new_doc))
        else:
            t = torch.as_tensor(new_doc)
            if t.device.type != "cpu" or t.numel() != bsz:
                raise ValueError("with lengths, new_doc is a bool or one host flag per video")
            nd = t.reshape(-1).to(torch.bool).numpy()
        eng = self._engine
        same = eng is not None and eng.has_state and eng.Bv == bsz
        mem = (eng._slots if eng._slots is not None else np.ones(bsz, bool)) if same else np.zeros(bsz, bool)
        hist = getattr(eng, "_hist", None)
        if same and hist is not None and hist.shape[1] != eng.H * ((Q + 31) // 32) and (mem & ~nd).any():
            raise ValueError(f"the number of queries changed inside a video ({Q} now): pass new_doc=True or keep Q")
        bad = (np.asarray(lens) > 0) & ~nd & ~mem
        if bad.any():
            raise ValueError(f"video slot(s) {np.flatnonzero(bad).tolist()} hold no memory and receive a chunk without "
                             "new_doc: pass new_doc for their first chunk")
        return lens, nd

    @torch.no_grad()
    def forward(self, k, q, new_doc, layer_n=None, u=None, generator=None, lengths=None):
        """lengths (variant 'gibbs'): per-video chunk lengths in frames (host ints, 0 = idle, else in [2, L]) of a
        ragged batch whose chunk k is padded to L frames; new_doc is then a bool or one host flag per video and is
        applied per slot (BatchedRectLTM.step), idle videos keep their memory and get zero rows."""
        if not k.is_cuda:
            raise RuntimeError("infinite_video_b200.LongTermAttention runs on CUDA tensors only (no CPU fallback)")
        lens = None
        if lengths is not None:
            lens, new_doc = self.check_ragged(k, lengths, new_doc, q.shape[1])
        self.device = k.device
        eng = self._get_engine(k.device)
        out_dtype = q.dtype
        # a 16-bit chunk (fp16 autocast in VideoChat2) is pooled straight from its storage: no up-cast pass
        # (variant R only: variant G consumes k un-pooled through the fp32 GEMMs)
        half_in = self.variant == "gibbs" and k.dtype in (torch.float16, torch.bfloat16)
        k32 = k.contiguous() if half_in else k.float().contiguous()
        q32 = q.float().contiguous()
        bsz = k32.size(0)
        if self.variant == "gibbs":
            self.length = k32.size(1) // self.tokens_per_frame            # gibbs:291-292
        if lens is None and new_doc:
            eng.reset()                                                    # gibbs:300-302
            sp = LongTermAttention._shared_pool
            if sp["key"] is None or sp["key"][0]() is not k:               # do not keep the last video's frames alive
                sp.update(key=None, x=None, k16=None)
        if eng.Bv is not None and eng.Bv != bsz:
            eng.reset()            # a different batch size starts from scratch: decide that BEFORE touching the RNG
        if eng.has_state and eng.sticky:
            if u is None:
                u = self._draw_uniforms(bsz, generator)
            u = u.to(k.device, torch.float64)
        else:
            u = None
        pooled = None
        # (a batch of idle videos has no frames: the step takes its empty chunk itself, no zero-size pooled tensor)
        if self.variant == "gibbs" and self.share_pooling and (lens is None or any(lens)):
            # identity of the tensor OBJECT (a weak reference) + its version counter: a data pointer alone is not
            # a key, the caching allocator hands the same address to the next chunk
            sp = LongTermAttention._shared_pool
            ref = sp["key"]
            hit = (ref is not None and ref[0]() is k and ref[1] == k._version and ref[2] == self.tokens_per_frame
                   and ref[3] == lens and sp["x"] is not None and sp["x"].device == k.device)
            if not hit:
                sp["x"], sp["k16"] = eng.pool(k32, lengths=lens), None
                sp["key"] = (weakref.ref(k), k._version, self.tokens_per_frame, lens)
            pooled = sp["x"]
        if lens is not None:
            ctx = eng.step(k32, q32, u=u, new_doc=torch.from_numpy(new_doc), pooled=pooled, lengths=lens)
        elif pooled is not None:
            ctx = eng.step(k32, q32, u=u, new_doc=False, pooled=pooled)
        else:
            ctx = eng.step(k32, q32, u=u, new_doc=False)
        if self.output_density and self.variant == "gibbs":
            self.alphas = eng.density()
            if self.dump_path is not None:
                import pickle
                with open(self.dump_path, "wb") as f:                      # gibbs:344-345
                    pickle.dump(self.alphas.cpu(), f)
        if self.kl_regularizer:                                            # gauss:296-304, :389-390
            self.kl_reg = eng.kl(self.mu_0, self.sigma_0)
            return ctx.to(out_dtype), self.kl_reg
        return ctx.to(out_dtype)

    def pool_for_caller(self, k, lengths=None):
        """One pass over an fp32 chunk for both halves of the caller's cross-attention branch: pools the frames for
        this (and every other) LTM layer -- the result is parked in the shared-pooling slot, so the following
        `forward(k, ...)` does not stream the chunk again -- and returns the chunk as float16 for the short-term
        attention GEMMs (cross_attention.py).  Every cross-attention layer of a Q-former is handed the same chunk: the
        second and later layers find both results in the slot.  `lengths` (ragged chunk): the frames are packed and
        the fp16 chunk is k16[Bv, ld16, e] padded per video (`BatchedRectLTM.pool`); the slot is keyed on the lengths
        too, so `forward(k, ..., lengths=)` with the same lengths finds it."""
        lens = None
        if lengths is not None:
            if self.variant != "gibbs":
                raise NotImplementedError("per-video lengths exist for variant 'gibbs' only")
            lens = _as_lengths(lengths, k.shape[0], k.shape[1] // self.tokens_per_frame)
        sp = LongTermAttention._shared_pool
        ref = sp["key"]
        if (ref is not None and ref[0]() is k and ref[1] == k._version and ref[2] == self.tokens_per_frame
                and ref[3] == lens and sp["x"] is not None and sp["k16"] is not None and sp["x"].device == k.device):
            return sp["k16"]
        eng = self._get_engine(k.device)
        pooled, k16 = eng.pool(k.contiguous(), with_half=True, lengths=lens)
        sp.update(key=(weakref.ref(k), k._version, self.tokens_per_frame, lens), x=pooled, k16=k16)
        return k16

    def extra_repr(self):
        return (f"variant={self.variant}, num_basis={self.attn_num_basis}, tau={self.tau}, "
                f"sticky={self.sticky_memories}, nb_samples={self.nb_samples}")
