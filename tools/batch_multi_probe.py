"""Several outputs per problem in a batch: per-problem times of the r-output batch (tgp_loglike_batch_multi value, and
tgp_loglike_grad_batch_multi value and gradient) against a loop of single tgp_loglike_multi / tgp_loglike_grad_multi
calls and against r separate single-output batch calls, over N x B x r; then the single-output batch
(tgp_loglike_batch, tgp_loglike_grad_batch) of this build against the same entries of another build of the library
(the parent commit's), alternated in the same process.

    python tools/batch_multi_probe.py [--out profiles/batch_multi_probe.json] [--parent-lib PATH] [--quick]

Every arm is timed with CUDA events around a window of back-to-back warmed calls holding at least --min-seconds of
work, the arms in turn, --reps times; medians per problem are reported with the spread (min, max) of the rounds.  The
backward sweep is timed on its own as the value call with want_alpha against without, N in {1000, 4000} x B in
{148, 512} x r in {2, 4, 8}: r = 4 runs one sweep CTA per problem, r = 8 two.  The single loop runs over the
first min(B, 16) problems (its per-problem cost does not depend on B).  Batches run as one call (budget 120 GB).
--parent-lib: a libtreegp_b200.so built from the parent commit (make in a checkout of it); without it the comparison
is skipped.  Card name, power limit and max SM clock are read in the same call."""
import argparse
import ctypes
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from batch_probe import card, problems  # noqa: E402

BUDGET = 120 << 30


def event_time(fn, n=1):
    """Seconds per call of fn over n back-to-back calls, from CUDA events around them."""
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(n):
        fn()
    e.record()
    e.synchronize()
    return s.elapsed_time(e) / 1e3 / n


def rounds(arms, reps, min_seconds):
    """{name: [seconds per call, one per round]}: every arm warmed by one timed call, which sets how many calls fill a
    window of min_seconds; then the arms in turn, reps times, one window each."""
    calls = {k: max(1, int(np.ceil(min_seconds / max(event_time(fn), 1e-7)))) for k, fn in arms.items()}
    t = {k: [] for k in arms}
    for _ in range(reps):
        for k, fn in arms.items():
            t[k].append(event_time(fn, calls[k]))
    return t


def stat(ts, per):
    us = np.array(ts) / per * 1e6
    return {"median": float(np.median(us)), "min": float(us.min()), "max": float(us.max())}


def grid_point(N, B, r, reps, min_seconds):
    from treegp_b200 import backend

    X, _, e2, descs = problems(N, B)
    rng = np.random.default_rng(1)
    Y = backend.to_device(rng.normal(size=(N * B, r)))
    cols = [Y[:, c].contiguous() for c in range(r)]
    sizes = [N] * B
    ns = min(B, 16)
    sums = [backend.as_sum(d) for d in descs]
    res = {}

    def single(grad):
        def run():
            for b in range(ns):
                s = slice(b * N, (b + 1) * N)
                if grad:
                    backend.loglike_grad(X[s], Y[s], e2[s], sums[b])
                else:
                    backend.loglike(X[s], Y[s], e2[s], sums[b])
        return run

    def batch(grad):
        fn = backend.loglike_grad_batch if grad else backend.loglike_batch

        def run():
            res[grad] = fn(X, Y, e2, sizes, descs, budget_bytes=BUDGET)[0]
        return run

    def separate(grad):
        fn = backend.loglike_grad_batch if grad else backend.loglike_batch

        def run():
            for c in range(r):
                fn(X, cols[c], e2, sizes, descs, budget_bytes=BUDGET)
        return run

    arms = {"batch_value": batch(False), "batch_grad": batch(True), "single_loop_value": single(False),
            "single_loop_grad": single(True), "separate_value": separate(False), "separate_grad": separate(True)}
    t = rounds(arms, reps, min_seconds)
    out = {"N": N, "B": B, "r": r, "reps": reps, "min_seconds": min_seconds, "single_problems_timed": ns}
    for k, v in t.items():
        out[k + "_us_per_problem"] = stat(v, ns if k.startswith("single") else B)
    m = lambda k: out[k + "_us_per_problem"]["median"]
    for kind in ("value", "grad"):
        out["speedup_%s_vs_single_loop" % kind] = m("single_loop_" + kind) / m("batch_" + kind)
        out["speedup_%s_vs_separate" % kind] = m("separate_" + kind) / m("batch_" + kind)
    # the joint value is the r-output likelihood of tgp_loglike_multi: check one problem against the single call
    o1 = backend.loglike(X[:N], Y[:N], e2[:N], sums[0])[0]
    out["value_bitwise_equal_problem0"] = bool(torch.equal(res[False][0], o1))
    return out


def parent_compare(parent_lib, N, B, reps, min_seconds):
    """tgp_loglike_batch and tgp_loglike_grad_batch of this build and of `parent_lib`, alternated."""
    from treegp_b200 import _cabi, backend

    libs = {"this": _cabi.load(), "parent": ctypes.CDLL(parent_lib)}
    X, y, e2, descs = problems(N, B)
    off = backend.batch_offsets([N] * B)
    ks = backend._ksum_array(descs)
    dev = X.device
    work = torch.empty(backend.batch_work_doubles([N] * B), dtype=torch.float64, device=dev)
    scratch = torch.empty(backend.grad_batch_scratch_doubles([N] * B), dtype=torch.float64, device=dev)
    alpha = torch.empty(N * B, dtype=torch.float64, device=dev)
    info = torch.empty(B, dtype=torch.int32, device=dev)
    outs = {}
    P = backend._p

    def value(name):
        def run():
            o = torch.empty((B, 3), dtype=torch.float64, device=dev)
            _cabi.check(libs[name].tgp_loglike_batch(P(X), P(y), P(e2), backend._host_i64(off), ctypes.c_int32(B),
                                                     ctypes.cast(ks, ctypes.c_void_p), P(work), P(alpha),
                                                     ctypes.c_int(0), P(o), P(info), P(None)))
            outs[("value", name)] = o
        return run

    def grad(name):
        def run():
            o = torch.empty((B, _cabi.GRAD_BATCH_OUT), dtype=torch.float64, device=dev)
            _cabi.check(libs[name].tgp_loglike_grad_batch(P(X), P(y), P(e2), backend._host_i64(off),
                                                          ctypes.c_int32(B), ctypes.cast(ks, ctypes.c_void_p), P(work),
                                                          P(alpha), P(o), P(info), P(scratch), P(None)))
            outs[("grad", name)] = o
        return run

    for lib in libs.values():
        for name in ("tgp_loglike_batch", "tgp_loglike_grad_batch"):
            getattr(lib, name).restype = ctypes.c_int
    arms = {"value_this": value("this"), "value_parent": value("parent"), "grad_this": grad("this"),
            "grad_parent": grad("parent")}
    t = rounds(arms, reps, min_seconds)
    out = {"N": N, "B": B, "reps": reps, "min_seconds": min_seconds}
    for k, v in t.items():
        out[k + "_us_per_problem"] = stat(v, B)
    for kind in ("value", "grad"):
        out[kind + "_bitwise_equal"] = bool(torch.equal(outs[(kind, "this")], outs[(kind, "parent")]))
        a, b = out[kind + "_this_us_per_problem"], out[kind + "_parent_us_per_problem"]
        out[kind + "_this_over_parent"] = a["median"] / b["median"]
        out[kind + "_ranges_overlap"] = a["min"] <= b["max"] and b["min"] <= a["max"]
    return out


def sweep_point(N, B, r, reps, min_seconds):
    """The backward sweep of tgp_loglike_batch_multi: the value call with want_alpha (K^-1 Y) against without (L^-1 Y).
    They differ by the sweep launch alone; every other launch is the same."""
    from treegp_b200 import backend

    X, _, e2, descs = problems(N, B)
    Y = backend.to_device(np.random.default_rng(2).normal(size=(N * B, r)))
    arms = {w: (lambda w=w: backend.loglike_batch(X, Y, e2, [N] * B, descs, want_alpha=w, budget_bytes=BUDGET))
            for w in (False, True)}
    t = rounds(arms, reps, min_seconds)
    off, on = (stat(t[w], B) for w in (False, True))
    return {"N": N, "B": B, "r": r, "reps": reps, "min_seconds": min_seconds, "no_sweep_us_per_problem": off,
            "with_sweep_us_per_problem": on, "sweep_us_per_problem": on["median"] - off["median"],
            "sweep_ctas_per_problem": -(-r // (1 if r == 1 else 2 if r == 2 else 4))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/batch_multi_probe.json")
    ap.add_argument("--parent-lib", default=None)
    ap.add_argument("--quick", action="store_true", help="two small points (a rehearsal)")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--min-seconds", type=float, default=0.2, help="work per timed window")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("batch_multi_probe needs a CUDA device")
    torch.cuda.set_device(0)
    rec = {"card": card(), "grid": [], "sweep": [], "parent": []}
    Ns, Bs, Rs = ([250], [16], [2]) if a.quick else ([250, 1000, 4000], [16, 148, 512], [2, 8])
    for N in Ns:
        for B in Bs:
            for r in Rs:
                p = grid_point(N, B, r, a.reps, a.min_seconds)
                rec["grid"].append(p)
                print(json.dumps(p), flush=True)
                torch.cuda.empty_cache()
    for N in ([250] if a.quick else [1000, 4000]):
        for B in ([16] if a.quick else [148, 512]):
            for r in ([2] if a.quick else [2, 4, 8]):
                p = sweep_point(N, B, r, a.reps, a.min_seconds)
                rec["sweep"].append(p)
                print(json.dumps(p), flush=True)
                torch.cuda.empty_cache()
    if a.parent_lib:
        for N in Ns:
            for B in Bs:
                p = parent_compare(a.parent_lib, N, B, 2 * a.reps, a.min_seconds)
                rec["parent"].append(p)
                print(json.dumps(p), flush=True)
                torch.cuda.empty_cache()
    rec["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(rec, f, indent=1)


if __name__ == "__main__":
    main()
