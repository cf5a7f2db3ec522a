#!/usr/bin/env python
"""Timing of the dense building blocks (CUDA events): gemm_nt_sub, potrf stages, trsv."""
import os, sys
import numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from treegp_b200 import backend

def timed(fn, reps=3):
    fn(); torch.cuda.synchronize(); ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); fn(); b.record(); torch.cuda.synchronize(); ts.append(a.elapsed_time(b) * 1e-3)
    return min(ts)

for (m, n, k, low) in [(20480, 20480, 512, 1), (20480, 20480, 512, 0), (40960, 512, 64, 0), (8192, 8192, 512, 1), (30000, 448, 64, 0)]:
    C = torch.zeros((m, backend.even(n)), dtype=torch.float64, device="cuda")
    A = torch.randn((m, k), dtype=torch.float64, device="cuda")
    B = torch.randn((n, k), dtype=torch.float64, device="cuda")
    t = timed(lambda: backend.gemm_nt_sub(C, m, n, A, B, k, lower_only=bool(low)))
    fl = 2.0 * m * n * k * (0.5 if low else 1.0)
    print("gemm m=%d n=%d k=%d lower=%d: %.3f ms  %.1f TF" % (m, n, k, low, t * 1e3, fl / t / 1e12), flush=True)
    del C, A, B
for n in [int(v) for v in os.environ.get("DP_N", "4096,10000,20000").split(",")]:
    A = torch.randn((n, 64), dtype=torch.float64, device="cuda")
    ws = backend.alloc_matrix(n, n)
    def fill():
        ws[:, :n] = (A @ A.T)
        ws[:, :n].diagonal().add_(float(n))
    fill(); torch.cuda.synchronize()
    keep = ws.clone()
    def chol():
        ws.copy_(keep); backend.potrf(ws, n)
    tc = timed(lambda: ws.copy_(keep))
    t = timed(chol) - tc
    tl = timed(lambda: torch.linalg.cholesky(keep[:, :n]))
    b = torch.randn(n, dtype=torch.float64, device="cuda")
    ts = timed(lambda: backend.potrs_vec(ws, n, b.clone()))
    print("potrf n=%d: %.2f ms  %.1f TF | cusolver %.2f ms %.1f TF | potrs_vec %.2f ms (%.0f GB/s)" % (
        n, t * 1e3, n ** 3 / 3 / t / 1e12, tl * 1e3, n ** 3 / 3 / tl / 1e12, ts * 1e3, 8.0 * n * n / ts / 1e9), flush=True)
    del ws, keep, A
