"""Timing of the envelope factorisation against the dense one (one GPU): configs[2] (N = 40k AnisotropicVonKarman,
field 160, size 1.5) and configs[1] (N = 10k AnisotropicRBF, field 63, size 0.5).  CUDA events, 3 repetitions."""
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench  # noqa: E402
import treegp_b200 as treegp  # noqa: E402
from treegp_b200 import backend  # noqa: E402
from treegp_b200.kernels import lower_kernel  # noqa: E402
from treegp_b200.two_pcf import get_correlation_length_matrix  # noqa: E402


def ev(fn, reps=3):
    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts))


def probe(name, X, kstr, noise):
    n = len(X)
    desc = lower_kernel(treegp.eval_kernel(kstr), 2)
    Xd = backend.as_points(X)
    plan = backend.plan_envelope(Xd, desc)
    rng = np.random.default_rng(0)
    y = backend.to_device(rng.normal(size=n))
    e2 = backend.to_device(np.full(n, noise ** 2))
    work = backend.alloc_matrix(n + 1, n)
    print("%s: N = %d, envelope %s" % (name, n, "not chosen" if plan is None else
          "axis %d, d_cut / extent = %.3f, flops %.3g of %.3g dense (%.1fx fewer)" % (
              plan["axis"], plan["dcut"] / (X[:, plan["axis"]].max() - X[:, plan["axis"]].min()), plan["flops"],
              plan["flops_dense"], plan["flops_dense"] / plan["flops"])))
    if plan is None:
        return
    o, re = plan["order"], plan["row_end"]
    Xs, ys, es = Xd[o].contiguous(), y[o].contiguous(), e2[o].contiguous()
    t_k = ev(lambda: backend.kmat_sym(Xs, desc, es, out=work, lower_only=True))

    def fac(row_end):
        backend.kmat_sym(Xs, desc, es, out=work, lower_only=True)
        backend.potrf(work, n, row_end=row_end)

    t_d, t_e = ev(lambda: fac(None)) - t_k, ev(lambda: fac(re)) - t_k
    print("  K build %.2f ms; potrf dense %.2f ms (%.1f TFLOP/s), envelope %.2f ms (%.1f TFLOP/s of its own flops): %.1fx"
          % (t_k, t_d, n ** 3 / 3 / t_d / 1e9, t_e, plan["flops"] / t_e / 1e9, t_d / t_e))
    for want in (False, True):
        td = ev(lambda: backend.loglike(Xs, ys, es, desc, work=work, want_alpha=want))
        te = ev(lambda: backend.loglike(Xs, ys, es, desc, work=work, want_alpha=want, row_end=re))
        od = backend.loglike(Xs, ys, es, desc, work=work, want_alpha=want)[0].cpu().numpy()
        oe = backend.loglike(Xs, ys, es, desc, work=work, want_alpha=want, row_end=re)[0].cpu().numpy()
        print("  tgp_loglike(want_alpha=%d): dense %.2f ms, envelope %.2f ms (%.1fx); logL %.12g vs %.12g (rel %.1e)"
              % (want, td, te, td / te, od[0], oe[0], abs(od[0] - oe[0]) / abs(od[0])))
    m = 4096
    Xt = backend.as_points(np.random.default_rng(1).uniform(X.min(0), X.max(0), size=(m, 2)))
    backend.potrf(backend.kmat_sym(Xs, desc, es, out=work, lower_only=True), n, row_end=re)
    V = backend.kmat_cross(Xt, Xs, desc)
    V0 = V.clone()
    td = ev(lambda: (V.copy_(V0), backend.trsm_rows(work, n, V, m)))
    te = ev(lambda: (V.copy_(V0), backend.trsm_rows(work, n, V, m, row_end=re)))
    tc = ev(lambda: V.copy_(V0))
    print("  trsm_rows, %d right-hand sides: dense %.2f ms, envelope %.2f ms (%.1fx)" % (m, td - tc, te - tc, (td - tc) / (te - tc)))


def main():
    X, _, kstr, _, _, noise, _ = bench.gp_problem(int(os.environ.get("PN", "40000")), 16)
    probe("configs[2]", X, kstr, noise)
    rng = np.random.default_rng(7)
    n = 10_000
    L = 80.0 * np.sqrt(n / 16000.0)
    inv = np.linalg.inv(get_correlation_length_matrix(0.5, 0.2, 0.2))
    kstr = "4.0 * AnisotropicRBF(invLam=array([[%.17g, %.17g], [%.17g, %.17g]]))" % (inv[0, 0], inv[0, 1], inv[1, 0], inv[1, 1])
    probe("configs[1]", rng.uniform(-L / 2, L / 2, size=(n, 2)), kstr, 0.01)


if __name__ == "__main__":
    main()
