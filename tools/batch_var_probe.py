"""Predictive variance and leave-one-out predictions of many independent small problems: a warmed loop of single dense
calls against one batched call, over N x B with M = 1000 test points per problem.

    python tools/batch_var_probe.py [--out profiles/batch_var_probe.json] [--quick]

Variance arms: a loop of tgp_loglike_sum + tgp_predict_var_sum (dense) per problem, against one
backend.predict_var_batch call (tgp_loglike_batch + tgp_predict_var_batch).  LOO arms: a loop of
GPInterpolation.loo_predict (BANDED_SOLVE = False) per problem, against one backend.loo_batch call with its results
copied to the host, as loo_predict copies its own.  Per point the four arms are timed in turn, each with CUDA events
around a warmed pass, --reps times; the medians are reported per problem.  The single loops run over the first
min(B, 16) problems (their per-problem cost does not depend on B).  The batches run as one call (budget 96 GB).  The
single results are compared with the batch's in the same run.  Card name, power limit and max SM clock are read in the
same call."""
import argparse
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from batch_probe import card, problems  # noqa: E402

BUDGET = 96 << 30
M = 1000


def event_time(fn):
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    fn()
    e.record()
    e.synchronize()
    return s.elapsed_time(e) / 1e3


def grid_point(N, B, reps):
    from treegp_b200 import GPInterpolation, backend

    X, y, e2, descs = problems(N, B)
    rng = np.random.default_rng(1)
    Xs = backend.to_device(rng.uniform(0, np.sqrt(N) * 1.5, size=(M * B, 2)))
    sums = [backend.as_sum(d) for d in descs]
    work = backend.alloc_matrix(N + 1, N)
    ns = min(B, 16)
    Xh, yh, eh = X.cpu().numpy(), y.cpu().numpy(), np.sqrt(e2.cpu().numpy())
    gps = []
    for b in range(ns):
        gp = GPInterpolation(kernel="1.5 * AnisotropicRBF(invLam=array([[%.3f, 0.1], [0.1, 0.8]]))" % (0.4 + 0.001 * b),
                             optimizer="none", normalize=False)
        gp.initialize(Xh[b * N:(b + 1) * N], yh[b * N:(b + 1) * N], y_err=eh[b * N:(b + 1) * N])
        gps.append(gp)
    res = {}

    def single_var():
        for b in range(ns):
            r = slice(b * N, (b + 1) * N)
            backend.loglike(X[r], y[r], e2[r], sums[b], work=work)
            res[("sv", b)] = backend.predict_var(Xs[b * M:(b + 1) * M], X[r], sums[b], work)

    def batch_var():
        res["bv"] = backend.predict_var_batch(Xs, [M] * B, X, y, e2, [N] * B, descs, budget_bytes=BUDGET)

    def single_loo():
        for b in range(ns):
            res[("sl", b)] = gps[b].loo_predict()

    def batch_loo():
        mean, var, info = backend.loo_batch(X, y, e2, [N] * B, descs, budget_bytes=BUDGET)
        res["bl"] = (mean.cpu().numpy(), var.cpu().numpy(), info.cpu().numpy())

    old = GPInterpolation.BANDED_SOLVE
    GPInterpolation.BANDED_SOLVE = False
    try:
        arms = (single_var, batch_var, single_loo, batch_loo)
        for fn in arms:   # warm every arm
            fn()
        torch.cuda.synchronize()
        t = {fn.__name__: [] for fn in arms}
        for _ in range(reps):
            for fn, n in zip(arms, (ns, B, ns, B)):
                t[fn.__name__].append(event_time(fn) / n)
    finally:
        GPInterpolation.BANDED_SOLVE = old
    var, info = res["bv"]
    var_equal = all(torch.equal(var[b * M:(b + 1) * M], res[("sv", b)]) for b in range(ns))
    mean_l, var_l, info_l = res["bl"]
    loo_var_rel = max(float(np.max(np.abs(var_l[b * N:(b + 1) * N] - res[("sl", b)][1]) / np.abs(res[("sl", b)][1])))
                      for b in range(ns))
    loo_mean_rel = max(float(np.max(np.abs(mean_l[b * N:(b + 1) * N] - res[("sl", b)][0]))
                             / np.max(np.abs(res[("sl", b)][0]))) for b in range(ns))
    med = {k: float(np.median(v)) for k, v in t.items()}
    return {"N": N, "B": B, "M": M,
            "single_var_us_per_problem": med["single_var"] * 1e6, "batch_var_us_per_problem": med["batch_var"] * 1e6,
            "speedup_var": med["single_var"] / med["batch_var"],
            "single_loo_us_per_problem": med["single_loo"] * 1e6, "batch_loo_us_per_problem": med["batch_loo"] * 1e6,
            "speedup_loo": med["single_loo"] / med["batch_loo"],
            "single_problems_timed": ns, "reps": reps, "info_all_zero": bool(np.all(info.cpu().numpy() == 0)
                                                                                and np.all(info_l == 0)),
            "var_bitwise_equal": bool(var_equal), "loo_var_max_rel_diff": loo_var_rel,
            "loo_mean_max_rel_diff": loo_mean_rel}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/batch_var_probe.json")
    ap.add_argument("--quick", action="store_true", help="two small points (a rehearsal)")
    ap.add_argument("--reps", type=int, default=3)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("batch_var_probe needs a CUDA device")
    torch.cuda.set_device(0)
    rec = {"card": card(), "grid": []}
    pts = [(250, 16), (500, 16)] if a.quick else [(N, B) for N in (250, 500, 1000, 2000, 4000) for B in (16, 148, 512)]
    for N, B in pts:
        r = grid_point(N, B, a.reps)
        rec["grid"].append(r)
        print(json.dumps(r), flush=True)
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(rec, f, indent=1)


if __name__ == "__main__":
    main()
