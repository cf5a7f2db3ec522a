import ctypes, os, subprocess, sys
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
so = "/tmp/libtgp_trsv_timing.so"
srcs = ["kmat.cu", "dense.cu", "trsv.cu", "predict.cu", "pairbin.cu", "microbench.cu", "hostrng.cu", "vcorr.cu"]
subprocess.check_call(["/usr/local/cuda/bin/nvcc", "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a",
                       "-DTGP_TRSV_TIMING", "-Xcompiler", "-fPIC", "-shared", "-o", so] +
                      [os.path.join(ROOT, "treegp_b200/csrc", f) for f in srcs])
lib = ctypes.CDLL(so)
vp, i64 = ctypes.c_void_p, ctypes.c_int64
lib.tgp_trsv_only.argtypes = [vp, i64, i64, vp, ctypes.c_int, vp]
lib.tgp_device_error.argtypes = [ctypes.c_int]
n, which = int(sys.argv[1]), int(sys.argv[2])
ws = torch.randn((n, n + (n & 1)), dtype=torch.float64, device="cuda") * (0.5 / np.sqrt(n))
ws[:, :n].diagonal().fill_(1.5)
b = torch.randn(n, dtype=torch.float64, device="cuda")
bb = b.clone()
print("launch n=%d which=%d" % (n, which), flush=True)
rc = lib.tgp_trsv_only(ws.data_ptr(), n, ws.stride(0), bb.data_ptr(), which, None)
print("rc", rc, flush=True)
torch.cuda.synchronize()
print("done; device error", lib.tgp_device_error(0), flush=True)
Lm = torch.tril(ws[:, :n])
ref = torch.linalg.solve_triangular(Lm if which == 1 else Lm.T, b[:, None], upper=(which != 1))[:, 0]
print("max err", float((bb - ref).abs().max()), flush=True)
