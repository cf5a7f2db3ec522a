"""Sum kernels on the B200: one run, one JSON line in --outdir (kernel_sum_probe.json).

  * configs[2] geometry (N = 40k, the AnisotropicVonKarman of bench.py gp_problem, points in a 160 x 160 field):
    the K build, tgp_loglike_sum inside the envelope and tgp_loglike_grad_sum, each for the single-term entry, the same
    kernel as a one-term sum (expected: equal outputs and times) and VK + RBF + White.  CUDA events, the variants
    alternated, five rounds after a warm-up of each.
  * the truncated mean at M = 1e6 test points for the same three descriptors (backend.predict_mean, Hilbert sort
    included).
  * configs[1] size (N = 10k): the GPInterpolation log-likelihood fit of c * AnisotropicRBF + WhiteKernel with scipy's
    forward-difference gradient and with log_likelihood.ANALYTIC_GRADIENT, alternated twice after a warm-up of each:
    wall time, device evaluations, theta-hat and logL.

Prints the card's name, power limit and max SM clock first; they belong beside every number of the record.
Usage: python tools/kernel_sum_probe.py --outdir DIR
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
    except Exception as e:  # the record still says what it could not read
        out = "unknown (%s)" % e
    return out


def event_ms(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b)


def alternate(fns, rounds=5):
    """{name: [ms per round]} with the variants alternated inside every round, after one warm-up call of each."""
    for f in fns.values():
        f()
    torch.cuda.synchronize()
    out = {k: [] for k in fns}
    for _ in range(rounds):
        for k, f in fns.items():
            out[k].append(event_ms(f))
    return out


def as_sum(desc):
    from treegp_b200 import _cabi

    d = _cabi.TgpKernelSum()
    d.nterms, d.ndim, d.white = 1, desc.ndim, 0.0
    d.term[0] = desc
    return d


def cfg2(treegp, backend):
    from treegp_b200.kernels import lower_kernel, lower_kernel_sum
    from treegp_b200.two_pcf import get_correlation_length_matrix

    n = 40_000
    L = 160.0 * np.sqrt(n / 40000.0)
    inv = np.linalg.inv(get_correlation_length_matrix(1.5, 0.2, 0.2))
    vk = "AnisotropicVonKarman(invLam=array([[%.17g, %.17g], [%.17g, %.17g]]))" % (inv[0, 0], inv[0, 1], inv[1, 0],
                                                                                 inv[1, 1])
    k1 = "4.0 * " + vk
    k3 = "4.0 * %s + 0.5 * RBF(1.5) + WhiteKernel(1e-3)" % vk
    rng = np.random.default_rng(42)
    X = rng.uniform(-L / 2, L / 2, size=(n, 2))
    y, y_err = treegp.sample_grf(treegp.eval_kernel(k1), X, noise=0.01, seed=5)
    ll = treegp.log_likelihood(X, y, y_err)
    Xd, yd, e2, work = ll._device_state()
    d1 = lower_kernel(treegp.eval_kernel(k1), 2)
    descs = {"single": d1, "sum1": as_sum(d1), "vk_rbf_white": lower_kernel_sum(treegp.eval_kernel(k3), 2)}
    inputs = {k: ll._envelope_inputs(d) for k, d in descs.items()}
    rec = {"n": n, "kernel_single": k1, "kernel_sum": k3,
           "envelope_rows_mean": {k: float(np.mean(v[3] - np.minimum(np.arange(512, n + 512, 512), n)))
                                  for k, v in inputs.items()}}
    kbuf = backend.alloc_matrix(n, n, Xd.device)
    rec["kmat_sym_ms"] = alternate({k: (lambda d=d, i=inputs[k]: backend.kmat_sym(i[0], d, i[2], out=kbuf,
                                                                                 lower_only=True))
                                    for k, d in descs.items()})
    del kbuf
    rec["loglike_env_ms"] = alternate({k: (lambda d=d, i=inputs[k]: backend.loglike(i[0], i[1], i[2], d, work=work,
                                                                                   row_end=i[3]))
                                       for k, d in descs.items()})
    rec["loglike_grad_env_ms"] = alternate({k: (lambda d=d, i=inputs[k]: backend.loglike_grad(i[0], i[1], i[2], d,
                                                                                             work=work, row_end=i[3]))
                                            for k, d in descs.items()})
    outs = {k: backend.loglike_grad(i[0], i[1], i[2], descs[k], work=work, row_end=i[3])[0].cpu().numpy()
            for k, i in inputs.items()}
    rec["one_term_sum_grad_bit_identical"] = bool(np.array_equal(outs["single"], outs["sum1"][:7]))
    rec["logL"] = {k: float(v[0]) for k, v in outs.items()}
    rec["grad"] = {k: [float(x) for x in v[3:]] for k, v in outs.items()}
    # truncated mean, M = 1e6 test points in the same field
    alpha = torch.as_tensor(rng.normal(size=n), device=Xd.device)
    Xs = backend.as_points(rng.uniform(-L / 2, L / 2, size=(1_000_000, 2)))
    means = {}
    rec["predict_mean_trunc_M1e6_ms"] = alternate(
        {k: (lambda d=d, k=k: means.__setitem__(k, backend.predict_mean(Xs, Xd, d, alpha, truncate=True)))
         for k, d in descs.items()}, rounds=3)
    rec["one_term_sum_mean_bit_identical"] = bool(torch.equal(means["single"], means["sum1"]))
    return rec


def fit_cfg1(treegp, llmod, analytic):
    from treegp_b200.two_pcf import get_correlation_length_matrix

    rng = np.random.default_rng(7)
    n = 10_000
    L = 80.0 * np.sqrt(n / 16000.0)
    inv = np.linalg.inv(get_correlation_length_matrix(0.5, 0.2, 0.2))
    rbf = "AnisotropicRBF(invLam=array([[%.17g, %.17g], [%.17g, %.17g]]))" % (inv[0, 0], inv[0, 1], inv[1, 0], inv[1, 1])
    X = rng.uniform(-L / 2, L / 2, size=(n, 2))
    y, y_err = treegp.sample_grf(treegp.eval_kernel("4.0 * " + rbf), X, noise=0.01, seed=8)
    y = y + rng.normal(scale=0.1, size=n)            # white level 0.01 on top of the measurement errors
    kstr = "3.0 * %s + WhiteKernel(0.003)" % rbf
    llmod.log_likelihood.ANALYTIC_GRADIENT = analytic
    try:
        gp = treegp.GPInterpolation(kernel=kstr, optimizer="log-likelihood", normalize=True)
        gp.initialize(X, y, y_err=y_err)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        gp.solve()
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
    finally:
        llmod.log_likelihood.ANALYTIC_GRADIENT = False
    o = gp._optimizer
    return {"kernel_start": kstr, "white_true": 0.01, "fit_s": dt, "evaluations": int(o.n_evaluations),
            "theta": [float(v) for v in gp.kernel.theta], "logL": float(o._logL)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--outdir", required=True)
    args = ap.parse_args()
    os.makedirs(args.outdir, exist_ok=True)
    gpu = card()
    print("card (name, power.limit, clocks.max.sm):", gpu, flush=True)
    import treegp_b200 as treegp
    from treegp_b200 import backend
    llmod = sys.modules["treegp_b200.log_likelihood"]

    rec = {"card": gpu, "cfg2_N40k": cfg2(treegp, backend)}
    print(json.dumps(rec["cfg2_N40k"]), flush=True)
    rec["cfg1_fit"] = {}
    fit_cfg1(treegp, llmod, False)   # warm-up of both paths
    fit_cfg1(treegp, llmod, True)
    for _ in range(2):
        for analytic in (False, True):
            rec["cfg1_fit"].setdefault("analytic" if analytic else "fd", []).append(fit_cfg1(treegp, llmod, analytic))
    line = json.dumps(rec)
    print(line)
    with open(os.path.join(args.outdir, "kernel_sum_probe.json"), "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
