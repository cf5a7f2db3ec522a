"""Throughput of many independent small likelihood evaluations: B single dense tgp_loglike calls against one
tgp_loglike_batch, over N x B, plus a whole fit (GPInterpolationBatch against a loop of GPInterpolation).

    python tools/batch_probe.py [--out profiles/batch_probe.json] [--quick]

Times are CUDA-event times of warmed loops with at least --min-seconds of work per point.  The logL values of both
paths are compared bit for bit in the same run.  The achieved rate sum N^3/3 / t is set against the DMMA micro-peak
(tgp_microbench_fp64(1)).  Card name, power limit and SM clock are read in the same call."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def card():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        txt = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        txt = "unavailable (%s)" % e
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q + ": " + txt}


def problems(N, B, seed=0):
    from treegp_b200 import backend, eval_kernel
    from treegp_b200.kernels import lower

    rng = np.random.default_rng(seed)
    side = np.sqrt(N) * 1.5
    X = backend.to_device(rng.uniform(0, side, size=(N * B, 2)))
    y = backend.to_device(rng.normal(size=N * B))
    e2 = backend.to_device(rng.uniform(0.05, 0.1, size=N * B) ** 2)
    descs = [lower(eval_kernel("1.5 * AnisotropicRBF(invLam=array([[%.3f, 0.1], [0.1, 0.8]]))" % (0.4 + 0.001 * b)), 2)
             for b in range(B)]
    return X, y, e2, descs


def timed(fn, min_seconds):
    fn()
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps, total = 0, 0.0
    while total < min_seconds * 1e3:
        s.record()
        fn()
        e.record()
        e.synchronize()
        total += s.elapsed_time(e)
        reps += 1
    return total / reps / 1e3, reps


def grid_point(N, B, min_seconds):
    from treegp_b200 import backend

    X, y, e2, descs = problems(N, B)
    work = backend.alloc_matrix(N + 1, N)
    singles = {}

    def run_single():
        for b in range(B):
            r = slice(b * N, (b + 1) * N)
            singles[b] = backend.loglike(X[r], y[r], e2[r], descs[b], work=work, want_alpha=False)[0]

    res = {}

    def run_batch():
        res["out"] = backend.loglike_batch(X, y, e2, [N] * B, descs)[0]

    t_single, n_single = timed(run_single, min_seconds)
    t_batch, n_batch = timed(run_batch, min_seconds)
    ref = torch.stack([singles[b] for b in range(B)])
    equal = bool(torch.equal(ref, res["out"]))
    flop = B * N ** 3 / 3.0
    return {"N": N, "B": B, "t_single_loop_s": t_single, "t_batch_s": t_batch,
            "us_per_problem_single": 1e6 * t_single / B, "us_per_problem_batch": 1e6 * t_batch / B,
            "speedup": t_single / t_batch, "reps_single": n_single, "reps_batch": n_batch,
            "rate_single_tflops": flop / t_single / 1e12, "rate_batch_tflops": flop / t_batch / 1e12,
            "logL_bitwise_equal": equal}


def whole_fit(B, N, banded):
    from treegp_b200 import GPInterpolation, GPInterpolationBatch, log_likelihood

    rng = np.random.default_rng(1)
    Xs = [rng.uniform(-15, 15, size=(N, 2)) for _ in range(B)]
    ys = [np.sin(X[:, 0] / 3.0) * np.cos(X[:, 1] / 4.0) + rng.normal(scale=0.1, size=N) for X in Xs]
    es = [np.full(N, 0.1) for _ in range(B)]
    k = "0.6 * AnisotropicRBF(invLam=array([[0.06, 0.0], [0.0, 0.07]]))"
    log_likelihood.BANDED, GPInterpolation.BANDED_SOLVE = banded, banded
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    thetas = []
    for b in range(B):
        gp = GPInterpolation(kernel=k, optimizer="log-likelihood")
        gp.initialize(Xs[b], ys[b], y_err=es[b])
        gp.solve()
        thetas.append(gp.kernel.theta)
    torch.cuda.synchronize()
    t_loop = time.perf_counter() - t0
    t0 = time.perf_counter()
    gpb = GPInterpolationBatch(kernel=k, optimizer="log-likelihood")
    gpb.initialize(Xs, ys, es)
    gpb.solve()
    torch.cuda.synchronize()
    t_batch = time.perf_counter() - t0
    log_likelihood.BANDED, GPInterpolation.BANDED_SOLVE = True, True
    same = all(np.array_equal(thetas[b], gpb.kernels[b].theta) for b in range(B))
    return {"B": B, "N": N, "envelope_allowed": banded, "t_loop_s": t_loop, "t_batch_s": t_batch,
            "speedup": t_loop / t_batch, "theta_array_equal": same}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/batch_probe.json")
    ap.add_argument("--min-seconds", type=float, default=1.0)
    ap.add_argument("--quick", action="store_true")
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs a GPU"
    from treegp_b200 import backend

    rec = {"card": card(), "dmma_peak_tflops": backend.microbench_fp64(1), "grid": [], "fit": []}
    Ns, Bs = ([250, 1000], [1, 148]) if a.quick else ([250, 500, 1000, 2000, 4000], [1, 16, 148, 512])
    for N in Ns:
        for B in Bs:
            r = grid_point(N, B, a.min_seconds)
            print(json.dumps(r), flush=True)
            rec["grid"].append(r)
    for banded in (True, False):
        r = whole_fit(148 if not a.quick else 16, 1000, banded)
        print(json.dumps(r), flush=True)
        rec["fit"].append(r)
    rec["card_after"] = card()
    os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(rec, f, indent=1)


if __name__ == "__main__":
    main()
