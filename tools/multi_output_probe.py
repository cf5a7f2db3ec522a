"""Several outputs sharing one kernel on the B200: one run, one JSON line in --outdir (multi_output_probe.json).

  * configs[2] geometry (N = 40k, the AnisotropicVonKarman of bench.py gp_problem, points in a 160 x 160 field, the
    envelope factorisation): tgp_loglike_multi and tgp_loglike_grad_multi for r = 2 and 8 outputs against r
    single-output calls on the same data; and both triangular sweeps on the N = 40k factor for r = 1, 2, 4, 8 columns
    in one pass (tgp_potrs_multi) against r single-column solves (tgp_potrs_vec).  CUDA events, the arms alternated, five rounds after a warm-up of each.
  * the truncated mean at M = 1e6 test points for r = 2 and 8 (backend.predict_mean with alpha (N, r)) against r calls of
    backend.predict_mean (Hilbert sort included in both).
  * configs[1] size (N = 10k, c * AnisotropicRBF): the public fit ("log-likelihood", analytic gradient) plus predict at
    1e5 points of a 2-output field, against two single-output GPInterpolations; wall time, alternated twice after a
    warm-up of each.

Prints the card's name, power limit and max SM clock first; they belong beside every number of the record.
Usage: python tools/multi_output_probe.py --outdir DIR
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
    """{name: [ms per round]} with the arms alternated inside every round, after one warm-up call of each."""
    for f in fns.values():
        f()
    torch.cuda.synchronize()
    out = {k: [] for k in fns}
    for _ in range(rounds):
        for k, f in fns.items():
            out[k].append(event_ms(f))
    return out


def cfg2(treegp, backend):
    from treegp_b200.kernels import lower_kernel
    from treegp_b200.two_pcf import get_correlation_length_matrix

    n = 40_000
    L = 160.0 * np.sqrt(n / 40000.0)
    inv = np.linalg.inv(get_correlation_length_matrix(1.5, 0.2, 0.2))
    k1 = "4.0 * AnisotropicVonKarman(invLam=array([[%.17g, %.17g], [%.17g, %.17g]]))" % (inv[0, 0], inv[0, 1],
                                                                                        inv[1, 0], inv[1, 1])
    rng = np.random.default_rng(42)
    X = rng.uniform(-L / 2, L / 2, size=(n, 2))
    Y = rng.normal(size=(n, 8))
    ll = treegp.log_likelihood(X, Y, np.full(n, 0.1))
    _, _, _, work = ll._device_state()             # N + 8 rows
    d = lower_kernel(treegp.eval_kernel(k1), 2)
    Xo, Yo, eo, row_end = ll._envelope_inputs(d)
    rec = {"n": n, "kernel": k1}
    for r in (2, 8):
        Yr = Yo[:, :r].contiguous()
        cols = [Yr[:, c].contiguous() for c in range(r)]
        rec["loglike_env_r%d_ms" % r] = alternate({
            "multi": lambda: backend.loglike(Xo, Yr, eo, d, work=work, row_end=row_end),
            "singles": lambda: [backend.loglike(Xo, y, eo, d, work=work, row_end=row_end) for y in cols]})
        rec["loglike_grad_env_r%d_ms" % r] = alternate({
            "multi": lambda: backend.loglike_grad(Xo, Yr, eo, d, work=work, row_end=row_end),
            "singles": lambda: [backend.loglike_grad(Xo, y, eo, d, work=work, row_end=row_end) for y in cols]},
            rounds=3)
        m = backend.loglike(Xo, Yr, eo, d, work=work, row_end=row_end)[0].cpu().numpy()
        s = [float(backend.loglike(Xo, y, eo, d, work=work, row_end=row_end)[0][0].item()) for y in cols]
        rec["joint_logL_r%d" % r] = float(m[0])
        rec["sum_single_logL_r%d" % r] = float(sum(s))
    # both sweeps on the N = 40k factor (the whole triangle is read): r columns in one pass (tgp_potrs_multi) against
    # r single-column solves (tgp_potrs_vec), r = 1, 2, 4, 8
    backend.loglike(Xo, cols[0], eo, d, work=work, row_end=row_end)
    ld = work.stride(0)
    b = cols[0].clone()
    for r in (1, 2, 4, 8):
        B = torch.zeros((r, ld), dtype=torch.float64, device=Xo.device)
        B[:, :n] = Yo[:, :r].T
        rec["sweeps_both_N40k_r%d_ms" % r] = alternate({
            "multi": lambda B=B: backend.potrs_multi(work, n, B),
            "singles": lambda r=r: [backend.potrs_vec(work, n, b) for _ in range(r)]})
    # truncated mean, M = 1e6 test points in the same field
    alpha = torch.as_tensor(rng.normal(size=(n, 8)), device=Xo.device)
    Xs = backend.as_points(rng.uniform(-L / 2, L / 2, size=(1_000_000, 2)))
    for r in (2, 8):
        ar = alpha[:, :r].contiguous()
        acols = [ar[:, c].contiguous() for c in range(r)]
        res = {}
        rec["predict_mean_trunc_M1e6_r%d_ms" % r] = alternate({
            "multi": lambda: res.__setitem__("m", backend.predict_mean(Xs, Xo, d, ar, truncate=True)),
            "singles": lambda: res.__setitem__("s", [backend.predict_mean(Xs, Xo, d, a, truncate=True)
                                                     for a in acols])}, rounds=3)
        rec["predict_mean_trunc_r%d_columns_bit_identical" % r] = bool(all(
            torch.equal(res["m"][:, c], res["s"][c]) for c in range(r)))
    return rec


def fit_predict_cfg1(treegp, llmod, multi):
    from treegp_b200.two_pcf import get_correlation_length_matrix

    rng = np.random.default_rng(7)
    n = 10_000
    L = 80.0 * np.sqrt(n / 16000.0)
    inv = np.linalg.inv(get_correlation_length_matrix(0.5, 0.2, 0.2))
    rbf = "AnisotropicRBF(invLam=array([[%.17g, %.17g], [%.17g, %.17g]]))" % (inv[0, 0], inv[0, 1], inv[1, 0], inv[1, 1])
    X = rng.uniform(-L / 2, L / 2, size=(n, 2))
    y0, y_err = treegp.sample_grf(treegp.eval_kernel("4.0 * " + rbf), X, noise=0.01, seed=8)
    y1, _ = treegp.sample_grf(treegp.eval_kernel("4.0 * " + rbf), X, noise=0.01, seed=9)
    Y = np.stack([y0, y1], axis=1)
    Xs = rng.uniform(-L / 2, L / 2, size=(100_000, 2))
    kstr = "3.0 * " + rbf
    llmod.log_likelihood.ANALYTIC_GRADIENT = True
    try:
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        if multi:
            gps = [treegp.GPInterpolation(kernel=kstr, optimizer="log-likelihood", normalize=True)]
            gps[0].initialize(X, Y, y_err=y_err)
        else:
            gps = [treegp.GPInterpolation(kernel=kstr, optimizer="log-likelihood", normalize=True) for _ in range(2)]
            for c, gp in enumerate(gps):
                gp.initialize(X, Y[:, c], y_err=y_err)
        for gp in gps:
            gp.solve()
            gp.predict(Xs)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
    finally:
        llmod.log_likelihood.ANALYTIC_GRADIENT = False
    return {"fit_predict_s": dt, "evaluations": [int(gp._optimizer.n_evaluations) for gp in gps],
            "theta": [[float(v) for v in gp.kernel.theta] for gp in gps]}


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
    torch.cuda.empty_cache()
    fit_predict_cfg1(treegp, llmod, True)    # warm-up of both arms
    fit_predict_cfg1(treegp, llmod, False)
    rec["cfg1_two_outputs"] = {"multi": [], "two_singles": []}
    for _ in range(2):
        rec["cfg1_two_outputs"]["multi"].append(fit_predict_cfg1(treegp, llmod, True))
        rec["cfg1_two_outputs"]["two_singles"].append(fit_predict_cfg1(treegp, llmod, False))
    line = json.dumps(rec)
    print(line)
    with open(os.path.join(args.outdir, "multi_output_probe.json"), "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
