#!/usr/bin/env python
"""How fast does the frame pooling run beside each compute kernel?  (pool on a low-priority stream, kernel X
back-to-back on a high-priority stream for the whole duration)"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from infinite_video_b200 import ops, tables
dev = torch.device("cuda:0")
torch.manual_seed(0)
Bv, N, Q, D, H, L, T, E = 128, 256, 32, 768, 12, 256, 32, 768
tab = tables.rect_tables(L, N, .75); td = tab.to(dev)
k = torch.randn(Bv, L, T, E, device=dev)
Bc = torch.randn(Bv * N, E, device=dev)
Wkv = torch.randn(2 * D, E, device=dev) * 0.03; bkv = torch.randn(2 * D, device=dev) * 0.1
q = torch.randn(Bv, Q, D, device=dev)
KV = torch.empty(Bv * N, 2 * D, device=dev)
ops.project_kv_r(Bc, Wkv, bkv, out=KV)
KVv = KV.view(Bv, N, 2 * D)
xp = ops.pool_mean(k, 1)
B_past = torch.randn(Bv, N, E, device=dev)
idx = torch.randint(0, N, (Bv, 512), device=dev, dtype=torch.int32)
side = torch.cuda.Stream(device=dev, priority=0); comp = torch.cuda.Stream(device=dev, priority=-1)
def gemm(): ops.project_kv_r(Bc, Wkv, bkv, out=KV)
def attn(): ops.cont_attn_rect_tc(q, KVv, td["X"], td["W"], tab.W_out, tab.c_none, td["jb"], td["tb"])
def cons(): ops.consolidate_rect(B_past, xp, idx, None, td, N, L) if hasattr(ops, "consolidate_rect") else None
def t_alone(f, n=10):
    f(); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(True), torch.cuda.Event(True)
    e0.record(); [f() for _ in range(n)]; e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n
tp = t_alone(lambda: ops.pool_mean(k, 1))
print(f"pool alone {tp:.3f} ms")
for name, f in (("gemm", gemm), ("attention", attn)):
    tx = t_alone(f)
    reps = int(2.5 * tp / tx) + 2
    torch.cuda.synchronize()
    p0, p1 = torch.cuda.Event(True), torch.cuda.Event(True)
    c0, c1 = torch.cuda.Event(True), torch.cuda.Event(True)
    with torch.cuda.stream(comp):
        c0.record()
        for _ in range(reps): f()
        c1.record()
    with torch.cuda.stream(side):
        p0.record(); ops.pool_mean(k, 1); p1.record()
    torch.cuda.synchronize()
    tpc, txc = p0.elapsed_time(p1), c0.elapsed_time(c1) / reps
    print(f"{name:10s}: alone {tx:.3f} ms | beside pool {txc:.3f} ms ({txc/tx:.2f}x) | pool beside it {tpc:.3f} ms (speed {tp/tpc:.2f})")
