"""Value-and-gradient of many independent small problems: a warmed loop of single dense tgp_loglike_grad_sum calls
against one tgp_loglike_grad_batch call, over N x B, with the batch's value alone (tgp_loglike_batch) beside it; then
the lock-step fit of 148 problems of N = 1000 (AnisotropicRBF) with forward differences and with the analytic
gradient, against a loop of single analytic fits.

    python tools/batch_grad_probe.py [--out profiles/batch_grad_probe.json] [--quick]

Per point the three arms are timed in turn (single loop, batched value and gradient, batched value), each with CUDA
events around a warmed pass, --reps times; the medians are reported per problem.  The single loop runs over the first
min(B, 32) problems (its per-problem cost does not depend on B).  The batch runs as one call (budget 96 GB).  Card name,
power limit and max SM clock are read in the same call."""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from batch_probe import card, problems  # noqa: E402

BUDGET = 96 << 30


def event_time(fn):
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    fn()
    e.record()
    e.synchronize()
    return s.elapsed_time(e) / 1e3


def grid_point(N, B, reps):
    from treegp_b200 import backend

    X, y, e2, descs = problems(N, B)
    sums = [backend.as_sum(d) for d in descs]
    work = backend.alloc_matrix(N + 1, N)
    ns = min(B, 32)
    singles = {}

    def run_single():
        for b in range(ns):
            r = slice(b * N, (b + 1) * N)
            singles[b] = backend.loglike_grad(X[r], y[r], e2[r], sums[b], work=work)[0]

    res = {}

    def run_grad():
        res["grad"] = backend.loglike_grad_batch(X, y, e2, [N] * B, descs, budget_bytes=BUDGET)[0]

    def run_value():
        res["value"] = backend.loglike_batch(X, y, e2, [N] * B, descs, budget_bytes=BUDGET)[0]

    for fn in (run_single, run_grad, run_value):   # warm every arm
        fn()
    torch.cuda.synchronize()
    ts, tg, tv = [], [], []
    for _ in range(reps):
        ts.append(event_time(run_single) / ns)
        tg.append(event_time(run_grad) / B)
        tv.append(event_time(run_value) / B)
    ref = torch.stack([singles[b] for b in range(ns)])
    got = res["grad"][:ns, :ref.shape[1]]
    gerr = float(((got[:, 3:] - ref[:, 3:]).abs().max(dim=1).values / ref[:, 3:].abs().max(dim=1).values).max())
    lerr = float(((got[:, 0] - ref[:, 0]).abs() / ref[:, 0].abs()).max())
    t_s, t_g, t_v = (float(np.median(t)) for t in (ts, tg, tv))
    return {"N": N, "B": B, "single_grad_us_per_problem": t_s * 1e6, "batch_grad_us_per_problem": t_g * 1e6,
            "batch_value_us_per_problem": t_v * 1e6, "speedup_grad": t_s / t_g,
            "grad_over_value": t_g / t_v, "single_problems_timed": ns, "reps": reps,
            "max_rel_logL_diff": lerr, "max_rel_grad_diff": gerr}


def fit(B, N, seed=1):
    from treegp_b200 import GPInterpolation, GPInterpolationBatch, backend, log_likelihood

    rng = np.random.default_rng(seed)
    Xs, ys, es = [], [], []
    for _ in range(B):
        X = rng.uniform(-15, 15, size=(N, 2))
        Xs.append(X)
        ys.append(np.sin(X[:, 0] / 3.0) * np.cos(X[:, 1] / 4.0) + rng.normal(scale=0.1, size=N) + 0.3)
        es.append(rng.uniform(0.05, 0.1, size=N))
    kstr = "0.5 * AnisotropicRBF(invLam=array([[0.05, 0.0], [0.0, 0.08]]))"
    counts = {}
    wrapped = {}
    for name in ("loglike_batch", "loglike_grad_batch"):
        real = getattr(backend, name)

        def w(*a, _real=real, _name=name, **k):
            counts[_name] = counts.get(_name, 0) + 1
            return _real(*a, **k)
        wrapped[name] = (real, w)
        setattr(backend, name, w)
    old = (log_likelihood.ANALYTIC_GRADIENT, log_likelihood.BANDED, GPInterpolation.BANDED_SOLVE)
    log_likelihood.BANDED, GPInterpolation.BANDED_SOLVE = False, False
    out = {"B": B, "N": N, "kernel": kstr}
    thetas = {}
    try:
        for arm, analytic in (("batch_fd", False), ("batch_analytic", True)):
            log_likelihood.ANALYTIC_GRADIENT = analytic
            counts.clear()
            gpb = GPInterpolationBatch(kernel=kstr, optimizer="log-likelihood")
            gpb.initialize(Xs, ys, es)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            gpb.solve()
            torch.cuda.synchronize()
            out[arm] = {"seconds": time.perf_counter() - t0, "rounds": sum(counts.values())}
            thetas[arm] = np.array([k.theta for k in gpb.kernels])
        log_likelihood.ANALYTIC_GRADIENT = True
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        th = []
        for b in range(B):
            gp = GPInterpolation(kernel=kstr, optimizer="log-likelihood")
            gp.initialize(Xs[b], ys[b], y_err=es[b])
            gp.solve()
            th.append(gp.kernel.theta)
        torch.cuda.synchronize()
        out["single_analytic_loop"] = {"seconds": time.perf_counter() - t0}
        thetas["single"] = np.array(th)
    finally:
        log_likelihood.ANALYTIC_GRADIENT, log_likelihood.BANDED, GPInterpolation.BANDED_SOLVE = old
        for name, (real, _) in wrapped.items():
            setattr(backend, name, real)
    rel = lambda a, b: float(np.max(np.abs(a - b) / np.maximum(np.abs(b), 1e-300)))
    out["theta_max_rel_diff_batch_analytic_vs_single_analytic"] = rel(thetas["batch_analytic"], thetas["single"])
    out["theta_max_rel_diff_batch_analytic_vs_batch_fd"] = rel(thetas["batch_analytic"], thetas["batch_fd"])
    out["speedup_batch_analytic_vs_batch_fd"] = out["batch_fd"]["seconds"] / out["batch_analytic"]["seconds"]
    out["speedup_batch_analytic_vs_single_loop"] = (out["single_analytic_loop"]["seconds"]
                                                    / out["batch_analytic"]["seconds"])
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/batch_grad_probe.json")
    ap.add_argument("--quick", action="store_true", help="two small points and a small fit (a rehearsal)")
    ap.add_argument("--reps", type=int, default=3)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("batch_grad_probe needs a CUDA device")
    torch.cuda.set_device(0)
    rec = {"card": card(), "grid": []}
    pts = [(250, 16), (500, 16)] if a.quick else [(N, B) for N in (250, 500, 1000, 2000, 4000) for B in (16, 148, 512)]
    for N, B in pts:
        r = grid_point(N, B, a.reps)
        rec["grid"].append(r)
        print(json.dumps(r), flush=True)
    rec["fit"] = fit(8, 300) if a.quick else fit(148, 1000)
    print(json.dumps(rec["fit"]), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(rec, f, indent=1)


if __name__ == "__main__":
    main()
