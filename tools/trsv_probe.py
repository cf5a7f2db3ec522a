import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from treegp_b200 import backend
def timed(fn, reps=3):
    fn(); torch.cuda.synchronize(); ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); fn(); b.record(); torch.cuda.synchronize(); ts.append(a.elapsed_time(b) * 1e-3)
    return min(ts)
for n in (4096, 10000, 40000):
    ws = backend.alloc_matrix(n, n); ws.normal_(); ws[:, :n].diagonal().fill_(float(n))
    b = torch.randn(n, dtype=torch.float64, device="cuda")
    t = timed(lambda: backend.potrs_vec(ws, n, b.clone()))
    print("potrs_vec n=%d: %.2f ms (%.0f GB/s of 8 N^2 bytes)" % (n, t * 1e3, 8.0 * n * n / t / 1e9))
    del ws
