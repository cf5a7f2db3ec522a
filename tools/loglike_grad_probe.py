"""Analytic log-likelihood gradient on the B200: one run, one JSON line in --outdir.

  * configs[1] (N = 10k, 4.0 * AnisotropicRBF, generated as bench.py run_cfg2 does): the GPInterpolation
    log-likelihood fit with scipy's forward-difference gradient and with log_likelihood.ANALYTIC_GRADIENT, alternated
    twice after a warm-up of each: wall time, device evaluations, theta-hat and logL.
  * configs[2] size (N = 40k, AnisotropicVonKarman of bench.py gp_problem): one tgp_loglike_env against one
    tgp_loglike_grad (CUDA events), and tgp_selinv alone on the factor against its flop count from row_end.

Prints the card's name and power limit first; they belong beside every number of the record.
Usage: python tools/loglike_grad_probe.py --outdir DIR
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


def fit_cfg1(treegp, llmod, analytic):
    from treegp_b200.two_pcf import get_correlation_length_matrix

    rng = np.random.default_rng(7)
    n = 10_000
    L = 80.0 * np.sqrt(n / 16000.0)
    inv = np.linalg.inv(get_correlation_length_matrix(0.5, 0.2, 0.2))
    kstr = "4.0 * AnisotropicRBF(invLam=array([[%.17g, %.17g], [%.17g, %.17g]]))" % (inv[0, 0], inv[0, 1], inv[1, 0], inv[1, 1])
    X = rng.uniform(-L / 2, L / 2, size=(n, 2))
    kern = treegp.eval_kernel(kstr)
    y, y_err = treegp.sample_grf(kern, X, noise=0.01, seed=8)
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
    return {"fit_s": dt, "evaluations": int(o.n_evaluations), "theta": [float(v) for v in gp.kernel.theta],
            "logL": float(o._logL)}


def events_ms(fn, reps):
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return ts


def cfg2_timings(treegp, backend, reps=5):
    from treegp_b200.two_pcf import get_correlation_length_matrix

    n = 40_000
    L = 160.0 * np.sqrt(n / 40000.0)
    inv = np.linalg.inv(get_correlation_length_matrix(1.5, 0.2, 0.2))
    kstr = "%r**2 * AnisotropicVonKarman(invLam=array([[%.17g, %.17g], [%.17g, %.17g]]))" % (
        2.0, inv[0, 0], inv[0, 1], inv[1, 0], inv[1, 1])
    rng = np.random.default_rng(42)
    X = rng.uniform(-L / 2, L / 2, size=(n, 2))
    kern = treegp.eval_kernel(kstr)
    y, y_err = treegp.sample_grf(kern, X, noise=0.01, seed=5)
    ll = treegp.log_likelihood(X, y, y_err)
    Xd, yd, e2, work = ll._device_state()
    desc = treegp.kernels.lower_kernel(kern, 2)
    Xs, ys, es, re = ll._envelope_inputs(desc)
    v_ll = lambda: backend.loglike(Xs, ys, es, desc, work=work, row_end=re)
    v_gr = lambda: backend.loglike_grad(Xs, ys, es, desc, work=work, row_end=re)
    for f in (v_ll, v_gr):   # warm-up
        f()
    torch.cuda.synchronize()
    t_ll, t_gr = [], []
    for _ in range(reps):   # alternated
        t_ll += events_ms(v_ll, 1)
        t_gr += events_ms(v_gr, 1)
    # selinv alone: on a fresh factor every time (it works in place)
    t_si = []
    for _ in range(reps):
        backend.loglike(Xs, ys, es, desc, work=work, want_alpha=True, row_end=re)
        t_si += events_ms(lambda: backend.selinv(work, n, row_end=re), 1)
    out_g = v_gr()[0].cpu().numpy()
    out_l = v_ll()[0].cpu().numpy()
    f_si, f_fac = backend.selinv_flops(re, n), backend.envelope_flops(re, n)
    return {"n": n, "kernel": kstr, "row_end_blocks": len(re), "envelope_rows_mean": float(np.mean(re - np.minimum(
        np.arange(512, n + 512, 512), n))),
        "loglike_ms": t_ll, "loglike_grad_ms": t_gr, "selinv_ms": t_si,
        "selinv_flops": f_si, "factor_flops": f_fac, "selinv_over_factor_flops": f_si / f_fac,
        "selinv_tflops": f_si / (np.median(t_si) * 1e-3) / 1e12,
        "selinv_share_of_loglike_grad": float(np.median(t_si) / np.median(t_gr)),
        "loglike_grad_over_loglike": float(np.median(t_gr) / np.median(t_ll)),
        "logL_loglike": float(out_l[0]), "logL_loglike_grad": float(out_g[0]),
        "grad_ln_amp_m00_m01_m11": [float(v) for v in out_g[3:7]]}


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

    rec = {"card": gpu, "cfg1": {}}
    fit_cfg1(treegp, llmod, False)   # warm-up of both paths
    fit_cfg1(treegp, llmod, True)
    for rnd in range(2):
        for analytic in (False, True):
            rec["cfg1"].setdefault("analytic" if analytic else "fd", []).append(fit_cfg1(treegp, llmod, analytic))
    print(json.dumps(rec["cfg1"]), flush=True)
    rec["cfg2_N40k"] = cfg2_timings(treegp, backend)
    line = json.dumps(rec)
    print(line)
    with open(os.path.join(args.outdir, "loglike_grad_probe.json"), "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
