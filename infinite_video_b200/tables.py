"""Host-side constant tables of the LTM consolidation path.

Everything here depends only on ``(L, N, tau)`` (and the sigma set for the Gaussian variant) --
never on data -- so it is built once per shape on the host, cached, uploaded once, and reused
by every call / video.  The reference rebuilds the same information inside ``get_basis`` on
*every* forward (long_term_attention_gibbs.py:67-165, :298).

Why the host, and why torch CPU ops: membership of a position in a rectangular basis function is
decided by fp32 rounding of ``linspace``/``(edges[:-1]+edges[1:])/2``/``mu -+ width/2`` and the
half-open compare ``lo <= t < hi`` (basis_functions.py:227-266).  For non power-of-two ``N`` some
positions fall in *no* bin (SURVEY.md section 8a R3), so the integer tables must come from the very
same fp32 expressions, never from ``floor(t*N)``.  These are small integer/plan tables; no
per-call arithmetic happens here.

Variant R ("gibbs"): ``F F^T`` is diagonal (each position activates at most one indicator), hence
``G = F^T (F F^T + ridge I)^-1`` has at most one non-zero per row, ``1/(cnt_j + ridge)``.  The dense
ridge solve of the reference collapses to a segmented mean described by a CSR membership list.
"""
from dataclasses import dataclass, field
from functools import lru_cache

import numpy as np
import torch

NB_SAMPLES = 512          # long_term_attention_gibbs.py:55
RIDGE_PENALTY = 0.5       # :62
NB_STICKY_EDGES = 129     # :163
NUM_QUAD_POINTS = 1000    # :251 (expected_value default)


def _rect_bounds(n):
    """fp32 lower/upper bounds of the N indicator functions (gibbs:176-182, basis:248-249)."""
    edges = torch.linspace(0, 1, n + 1)
    mu = (edges[:-1] + edges[1:]) / 2
    width = torch.ones(n) / n
    return mu - width / 2, mu + width / 2


def rect_bin_of(t, n):
    """Index of the indicator active at each fp32 position (-1: none).  Raises if a position
    activates two indicators (then F F^T is not diagonal and the segmented-mean form is invalid)."""
    lo, hi = _rect_bounds(n)
    t = torch.as_tensor(t, dtype=torch.float32).reshape(-1, 1)
    hit = (t >= lo.unsqueeze(0)) & (t < hi.unsqueeze(0))
    nhit = hit.sum(1)
    if int(nhit.max()) > 1:
        raise NotImplementedError(
            f"num_basis={n}: a position activates two rectangular basis functions; the ridge system is "
            "not diagonal for this N")
    idx = hit.float().argmax(1)
    return torch.where(nhit > 0, idx, torch.full_like(idx, -1)).to(torch.int32)


def first_chunk_positions(l, spacing="linear"):
    """Padded frame positions of a first chunk (gibbs:103-110; `spacing='log'` :114-127: the L frame positions
    become e^{ln 2 * i / L} - 1, i = 1..L, between the same pads -- evaluated with the reference's own numpy / torch
    expression because bin membership is decided by its rounding)."""
    if l % 2:
        s = 1 / float(l)
        pos, trim = torch.linspace(-.5 + s, 1.5 - s, 2 * l - 1), (l - 1) // 2
    else:
        s = 1 / float(2 * l)
        pos, trim = torch.linspace(-.5 + s, 1.5 - s, 2 * l), l // 2
    if spacing == "log":
        mid = np.e ** (np.log(1 + 1) * torch.arange(1, l + 1) / l) - 1
        pos = torch.cat([pos[:int(l / 2)], mid.to(pos.dtype), pos[-int(l / 2):]])
    elif spacing != "linear":
        raise ValueError("spacing must be 'linear' or 'log'")
    return pos, trim


def update_positions(l, tau, nb_samples=NB_SAMPLES):
    """Padded positions of [S contracted samples | L new frames] (gibbs:134-150).
    Returns (all positions, number of left pads, sample positions)."""
    old = torch.arange(1, nb_samples + 1).float() * tau / nb_samples
    new = torch.arange(nb_samples + 1, l + nb_samples + 1).float()
    new = tau + (1 - tau) * (new - nb_samples) / l
    if l % 2:
        s = 1 / float(l + nb_samples)
        pad = torch.linspace(-.5 + s, 1.5 - s, 2 * (l + nb_samples) - 1)
    else:
        s = 1 / float(2 * l + nb_samples)
        pad = torch.linspace(-.5 + s, 1.5 - s, 2 * (l + nb_samples))
    left, right = pad[pad < 0], pad[pad > 1]
    tot = nb_samples + l
    trim = (tot - 1) // 2 if tot % 2 else tot // 2
    allpos = torch.cat([left, old, new, right], 0)
    if left.numel() != trim or allpos.numel() - 2 * trim != tot:
        raise NotImplementedError(f"pad/trim misalignment for L={l}: the reference would regress shifted rows")
    return allpos, trim, old


def sticky_edges():
    bins = torch.linspace(0, 1, NB_STICKY_EDGES)
    nudged = bins.clone()
    nudged[0] = -.000001       # gibbs:198
    nudged[-1] = 1.000001      # gibbs:199
    return bins, nudged


def _csr(member_bin, n):
    """member_bin[p] in [-1,n) -> (ptr[n+1], members) listing positions per bin in ascending order."""
    mb = np.asarray(member_bin)
    order = np.argsort(mb, kind="stable")
    order = order[mb[order] >= 0]
    counts = np.bincount(mb[mb >= 0], minlength=n)
    ptr = np.zeros(n + 1, dtype=np.int32)
    ptr[1:] = np.cumsum(counts)
    return ptr, order.astype(np.int32)


@dataclass
class RectTables:
    """Constant tables of variant R for one (L, N, tau).  All arrays are host numpy; ``.to(device)``
    uploads them once as torch tensors."""
    L: int
    N: int
    tau: float
    S: int
    # first chunk: B = G0^T x
    seg_ptr0: np.ndarray = None      # int32 [N+1]
    seg_mem0: np.ndarray = None      # int32 [nnz0]  frame indices
    g0: np.ndarray = None            # fp32  [N]     1/(cnt+ridge)
    # update: B = G_inf^T [xm ; x]
    seg_ptr1: np.ndarray = None      # int32 [N+1]
    seg_mem1: np.ndarray = None      # int32 [nnz1]  p < S: sample p ; p >= S: frame p-S
    g1: np.ndarray = None            # fp32  [N]
    jf: int = 0                      # first bin of the update tables that holds a new frame (bins below it hold
                                     # re-sampled memory only: their K|V follow from the previous K|V, consolidate.cu)
    # update tables with the new frames folded per bin (csrc/pool.cu: pool_bins_kernel): the frames of bin xb_row0 + r
    # are the consecutive frames [fbin_ptr[r], fbin_ptr[r+1]) and enter seg_mem1b as ONE member, id S + r
    xb_row0: int = 0
    xb_rows: int = 0                 # 0: the frames of some bin are not consecutive -> no folding
    fbin_ptr: np.ndarray = None      # int32 [xb_rows+1]
    seg_ptr1b: np.ndarray = None     # int32 [N+1]
    seg_mem1b: np.ndarray = None     # int32 [nnz1b]  p < S: sample p ; p >= S: bin sum p-S
    # sticky histogram (129 nudged edges) and sampling
    tb: np.ndarray = None            # fp32 [129] evaluation edges
    jb: np.ndarray = None            # int32 [129] basis index at each edge (-1 none)
    bins: np.ndarray = None          # fp32 [129] un-nudged edges (sample positions are bins[b])
    bin2basis: np.ndarray = None     # int32 [128] basis index of position bins[b]
    # quadrature of expected_value: r_j = W_j e^{S_j} / (sum_i W_i e^{S_i} + W_out)
    W: np.ndarray = None             # fp32 [N]
    W_out: float = 0.0
    X: np.ndarray = None             # fp32 [N,32] extra operand rows of the tensor-core attention (or None)
    X16: np.ndarray = None           # fp16 [N,64] the same table for the fp16 attention (csrc/attn_tc.cu)
    c_none: float = 0.0              # trapezoid node weight of the sticky edges outside every basis
    # uniform (non-sticky) resampling table: basis index of sample s (-1 none)  (gibbs:152-157,:212)
    idx_uniform: np.ndarray = None   # int32 [S]
    # density side-output of the Video-LLaMA copy (gibbs:328-335): 3 x 256 evaluation points
    jd: np.ndarray = None            # int32 [768] basis index at each point (-1 none)
    wd: np.ndarray = None            # fp32  [768] trapezoid weight of the point inside its own segment
    _dev: dict = field(default_factory=dict, repr=False)

    def to(self, device):
        key = str(device)
        if key not in self._dev:
            d = {}
            for name in ("seg_ptr0", "seg_mem0", "g0", "seg_ptr1", "seg_mem1", "g1", "tb", "jb", "bins",
                         "bin2basis", "W", "idx_uniform", "jd", "wd"):
                d[name] = torch.from_numpy(getattr(self, name)).to(device)
            for name in ("fbin_ptr", "seg_ptr1b", "seg_mem1b"):
                d[name] = torch.from_numpy(getattr(self, name)).to(device) if self.xb_rows > 0 else None
            d["X"] = torch.from_numpy(self.X).to(device) if self.X is not None else None
            d["X16"] = torch.from_numpy(self.X16).to(device) if self.X16 is not None else None
            self._dev[key] = d
        return self._dev[key]

    def dense_G0(self):
        """Dense [L,N] operator (for tests): G0[p,j] = g0[j] if frame p is in bin j."""
        G = np.zeros((self.L, self.N), np.float32)
        for j in range(self.N):
            G[self.seg_mem0[self.seg_ptr0[j]:self.seg_ptr0[j + 1]], j] = self.g0[j]
        return G

    def dense_Ginf(self):
        G = np.zeros((self.S + self.L, self.N), np.float32)
        for j in range(self.N):
            G[self.seg_mem1[self.seg_ptr1[j]:self.seg_ptr1[j + 1]], j] = self.g1[j]
        return G


def _fold_frames(t, fb):
    """Update tables with the new frames folded per bin.  fb[f] = bin of frame f (-1: outside every basis).  Possible
    when the frames of the bins [jf, N) are consecutive runs that follow each other without a gap (they are whenever the
    frame positions increase, i.e. for both spacings of the reference); the members of a bin keep their order: samples
    first, then the bin sum."""
    S, N = t.S, t.N
    if t.jf >= N:
        return
    rows = N - t.jf
    ptr = np.zeros(rows + 1, np.int64)
    seg_ptr, seg_mem = [0], []
    end = None                                   # one past the last frame folded so far
    for j in range(N):
        mem = t.seg_mem1[t.seg_ptr1[j]:t.seg_ptr1[j + 1]]
        fr = mem[mem >= S] - S
        seg_mem.extend(int(m) for m in mem[mem < S])
        if fr.size:
            if j < t.jf or not np.array_equal(fr, np.arange(fr[0], fr[0] + fr.size)):
                return
            if end is None:
                ptr[:j - t.jf + 1] = int(fr[0])
            elif int(fr[0]) != end:
                return                           # a gap (frames outside every basis) between two bins
            end = int(fr[0]) + fr.size
            seg_mem.append(S + (j - t.jf))
        if j >= t.jf and end is not None:
            ptr[j - t.jf + 1] = end
        seg_ptr.append(len(seg_mem))
    covered = np.zeros(fb.shape[0], bool)
    covered[ptr[0]:ptr[-1]] = True
    if end is None or not np.array_equal(covered, fb >= 0):
        return
    t.xb_row0, t.xb_rows = t.jf, rows
    t.fbin_ptr = ptr.astype(np.int32)
    t.seg_ptr1b = np.asarray(seg_ptr, np.int32)
    t.seg_mem1b = np.asarray(seg_mem, np.int32)


@lru_cache(maxsize=64)
def rect_tables(L: int, N: int, tau: float, S: int = NB_SAMPLES, num_quad: int = NUM_QUAD_POINTS,
                spacing: str = "linear") -> RectTables:
    if L < 2:
        raise ValueError("chunks of a single frame are not supported (the reference fails on L=1)")
    t = RectTables(L=L, N=N, tau=float(tau), S=S)
    ridge = torch.tensor(RIDGE_PENALTY)

    # --- first chunk (gibbs:99-131 + compute_G :68-84)
    pos0, trim0 = first_chunk_positions(L, spacing)
    b0 = rect_bin_of(pos0, N).numpy()
    cnt0 = np.bincount(b0[b0 >= 0], minlength=N)                      # counts include pad positions
    frames0 = b0[trim0:trim0 + L]
    assert frames0.shape[0] == L
    t.seg_ptr0, t.seg_mem0 = _csr(frames0, N)
    t.g0 = (1.0 / (torch.from_numpy(cnt0).float() + ridge)).numpy()

    # --- update (gibbs:134-160)
    pos1, trim1, old = update_positions(L, tau, S)
    b1 = rect_bin_of(pos1, N).numpy()
    cnt1 = np.bincount(b1[b1 >= 0], minlength=N)
    core1 = b1[trim1:trim1 + S + L]
    t.seg_ptr1, t.seg_mem1 = _csr(core1, N)
    t.g1 = (1.0 / (torch.from_numpy(cnt1).float() + ridge)).numpy()
    fb = core1[S:]
    t.jf = int(fb[fb >= 0].min()) if (fb >= 0).any() else N
    _fold_frames(t, fb)

    # --- sticky edges (gibbs:163,:197-199,:207-208)
    bins, nudged = sticky_edges()
    t.tb = nudged.numpy().copy()
    t.bins = bins.numpy().copy()
    t.jb = rect_bin_of(nudged, N).numpy()
    t.bin2basis = rect_bin_of(bins[:-1], N).numpy()

    # --- quadrature weights of the 1000-point trapezoid rule folded per basis (gibbs:251-286)
    tq = torch.linspace(0, 1, num_quad)
    jq = rect_bin_of(tq, N).numpy()
    dt = (tq[1:] - tq[:-1]).double().numpy()
    wt = np.zeros(num_quad)
    wt[:-1] += dt / 2
    wt[1:] += dt / 2
    W = np.zeros(N)
    np.add.at(W, jq[jq >= 0], wt[jq >= 0])
    t.W = W.astype(np.float32)
    t.W_out = float(wt[jq < 0].sum())

    # --- operand rows appended to V^T by the tensor-core attention (csrc/attn_tc.cu): with the un-normalised
    # weights e_j = W_j exp(S_j - m) as the other operand, row 0 (ones) yields the quadrature normaliser
    # sum_j e_j and rows 1+2 (hi + lo, each exact in tf32) the trapezoid integral of the sticky histogram,
    # Z = sum_i w_i E_i = sum_j c_j exp(S_j - m) + c_none exp(-m), c_j = sum of the node weights w_i of the
    # edges that fall into basis j (gibbs:197-202,:248), as sum_j (c_j / W_j) e_j.
    tbd = t.tb.astype(np.float64)
    wn = np.zeros(tbd.shape[0])
    wn[:-1] += np.diff(tbd) / 2
    wn[1:] += np.diff(tbd) / 2
    cj = np.zeros(N)
    np.add.at(cj, t.jb[t.jb >= 0], wn[t.jb >= 0])
    t.c_none = float(wn[t.jb < 0].sum())
    X = np.zeros((N, 32), dtype=np.float32)
    if (W > 0).all():
        ratio = (cj / W).astype(np.float32)
        hi = (ratio.view(np.uint32) & np.uint32(0xFFFFE000)).view(np.float32)
        X[:, 0] = 1.0
        X[:, 1] = hi
        X[:, 2] = (ratio.astype(np.float64) - hi.astype(np.float64)).astype(np.float32)
        t.X = X
        # fp16 flavour: 1, and c_j / W_j as hi + lo halves (22 bits between them), in a 64-column MN atom
        X16 = np.zeros((N, 64), dtype=np.float16)
        X16[:, 0] = 1.0
        X16[:, 1] = ratio.astype(np.float16)
        X16[:, 2] = (ratio.astype(np.float64) - X16[:, 1].astype(np.float64)).astype(np.float16)
        t.X16 = X16
    else:
        t.X = None                     # a basis without quadrature points: the tensor-core path is not used

    # --- uniform re-sampling table (gibbs:152-157): psi.evaluate(t/tau) for each contracted position
    t.idx_uniform = rect_bin_of(old / tau, N).numpy()

    # --- density side-output grid (gibbs:328-334): per segment, trapz weights from the actual fp32 spacings
    jd, wd = [], []
    for a, b in ((0.0, 0.25), (0.25, 0.5), (0.5, 1.0)):
        ts = torch.linspace(a, b, 256)
        jd.append(rect_bin_of(ts, N).numpy())
        d = (ts[1:] - ts[:-1]).double().numpy()
        w = np.zeros(256)
        w[:-1] += d / 2
        w[1:] += d / 2
        wd.append(w.astype(np.float32))
    t.jd = np.concatenate(jd).astype(np.int32)
    t.wd = np.concatenate(wd)
    return t


class RectBank:
    """The chunk-length dependent tables of variant R -- first-chunk and update segment tables, weights and jf -- for
    every chunk length up to `Lmax`, at fixed strides, so that a kernel selects the tables of a video from its length
    alone (ragged batches, `BatchedRectLTM.step(..., lengths=...)`):

      seg_ptr0 / seg_ptr1  int32 [Lmax+1, N+1]  absolute offsets into the concatenated seg_mem0 / seg_mem1
      seg_mem0 / seg_mem1  int32                entry L at mem0_off(L) = L(L-1)/2, mem1_off(L) = L*S + L(L-1)/2
      g0 / g1              fp32  [Lmax+1, N]
      jf                   int32 [Lmax+1]       (host only: the step derives its projected-row split from it)

    Entries are filled on first use from `rect_tables(L, ...)`, which stays the single source of bin membership, and
    uploaded to a device stream-ordered on the current stream, once per (device, L).  Every other table of variant R
    (sticky edges, quadrature, uniform re-sampling, density grid) does not depend on L."""

    def __init__(self, Lmax, N, tau, S=NB_SAMPLES, spacing="linear"):
        self.Lmax, self.N, self.tau, self.S, self.spacing = int(Lmax), int(N), float(tau), int(S), spacing
        n = self.Lmax + 1
        self.seg_ptr0 = np.zeros((n, N + 1), np.int32)
        self.seg_ptr1 = np.zeros((n, N + 1), np.int32)
        self.seg_mem0 = np.zeros(self.mem0_off(n), np.int32)
        self.seg_mem1 = np.zeros(self.mem1_off(n), np.int32)
        self.g0 = np.zeros((n, N), np.float32)
        self.g1 = np.zeros((n, N), np.float32)
        self.jf = np.zeros(n, np.int32)
        self.filled = set()
        self._dev = {}

    @staticmethod
    def mem0_off(L):
        return L * (L - 1) // 2                          # a first chunk of l frames has at most l members

    def mem1_off(self, L):
        return L * self.S + L * (L - 1) // 2             # an update of l frames has at most S + l members

    def fill(self, lengths):
        """Host entries for every length in `lengths` (0 = idle, skipped); returns the lengths newly filled."""
        new = sorted({int(L) for L in lengths} - self.filled - {0})
        for L in new:
            if not 2 <= L <= self.Lmax:
                raise ValueError(f"chunk length {L} outside [2, {self.Lmax}]")
            t = rect_tables(L, self.N, self.tau, self.S, spacing=self.spacing)
            o0, o1 = self.mem0_off(L), self.mem1_off(L)
            self.seg_ptr0[L] = t.seg_ptr0 + o0
            self.seg_mem0[o0:o0 + t.seg_mem0.size] = t.seg_mem0
            self.seg_ptr1[L] = t.seg_ptr1 + o1
            self.seg_mem1[o1:o1 + t.seg_mem1.size] = t.seg_mem1
            self.g0[L], self.g1[L], self.jf[L] = t.g0, t.g1, t.jf
            self.filled.add(L)
        return new

    def entry(self, L):
        """The tables of length L sliced back out of the bank (host): (seg_ptr0, seg_mem0, g0, seg_ptr1, seg_mem1, g1,
        jf), in the layout of `rect_tables`."""
        o0, o1 = self.mem0_off(L), self.mem1_off(L)
        p0, p1 = self.seg_ptr0[L] - o0, self.seg_ptr1[L] - o1
        return (p0, self.seg_mem0[o0:o0 + p0[-1]], self.g0[L], p1, self.seg_mem1[o1:o1 + p1[-1]], self.g1[L],
                int(self.jf[L]))

    def to(self, device, lengths):
        """Device arrays holding (at least) the entries of `lengths`.  Entries not on this device yet are copied on the
        current stream, consecutive lengths in one copy per array."""
        key = str(device)
        d = self._dev.get(key)
        if d is None:
            d = dict(done=set())
            for name in ("seg_ptr0", "seg_mem0", "g0", "seg_ptr1", "seg_mem1", "g1"):
                d[name] = torch.zeros(getattr(self, name).shape, dtype=torch.float32 if name[0] == "g" else torch.int32,
                                      device=device)
            self._dev[key] = d
        self.fill(lengths)
        todo = sorted({int(L) for L in lengths} - d["done"] - {0})
        runs = []
        for L in todo:
            if runs and runs[-1][1] == L:
                runs[-1][1] = L + 1
            else:
                runs.append([L, L + 1])
        for a, b in runs:
            for name in ("seg_ptr0", "g0", "seg_ptr1", "g1"):
                d[name][a:b].copy_(torch.from_numpy(getattr(self, name)[a:b]))
            d["seg_mem0"][self.mem0_off(a):self.mem0_off(b)].copy_(
                torch.from_numpy(self.seg_mem0[self.mem0_off(a):self.mem0_off(b)]))
            d["seg_mem1"][self.mem1_off(a):self.mem1_off(b)].copy_(
                torch.from_numpy(self.seg_mem1[self.mem1_off(a):self.mem1_off(b)]))
        d["done"].update(todo)
        return d


# ----------------------------------------------------------------------------------------------
# Variant G (Gaussian RBF): host side only provides positions / basis parameters; the design matrix
# and the ridge solve run on the device (csrc/ridge.cu).
# ----------------------------------------------------------------------------------------------
@dataclass
class GaussTables:
    L: int
    N: int
    tau: float
    S: int
    sigmas: tuple
    basis_mu: np.ndarray = None      # fp32 [N]   (long_term_attention.py:191-198, mu-major meshgrid)
    basis_sigma: np.ndarray = None   # fp32 [N]
    pos0: np.ndarray = None          # fp32 [P0]  padded first-chunk positions
    trim0: int = 0
    pos1: np.ndarray = None          # fp32 [P1]  padded update positions
    trim1: int = 0
    tb: np.ndarray = None            # fp32 [129] nudged edges
    bins: np.ndarray = None          # fp32 [129]
    old_over_tau: np.ndarray = None  # fp32 [S]   uniform re-sampling positions


@lru_cache(maxsize=64)
def gauss_tables(L: int, N: int, tau: float, sigmas=(0.005, 0.01), S: int = NB_SAMPLES,
                 spacing: str = "linear") -> GaussTables:
    if L % 2:
        raise ValueError("variant G: odd chunk lengths are broken upstream (long_term_attention.py:162-168)")
    ns = len(sigmas)
    if N % ns:
        N += ns - N % ns                                              # (:107-108)
    mu, sg = torch.meshgrid(torch.linspace(0, 1, N // ns), torch.Tensor(list(sigmas)), indexing="ij")
    pos0, trim0 = first_chunk_positions(L, spacing)
    pos1, trim1, old = update_positions(L, tau, S)
    bins, nudged = sticky_edges()
    return GaussTables(L=L, N=N, tau=float(tau), S=S, sigmas=tuple(sigmas),
                       basis_mu=mu.flatten().numpy().copy(), basis_sigma=sg.flatten().numpy().copy(),
                       pos0=pos0.numpy().copy(), trim0=trim0, pos1=pos1.numpy().copy(), trim1=trim1,
                       tb=nudged.numpy().copy(), bins=bins.numpy().copy(),
                       old_over_tau=(old / tau).numpy().copy())
