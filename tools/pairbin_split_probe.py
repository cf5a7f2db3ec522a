"""Two builds of the library compared on the bench.py 2PCF workload: one JSON file in --outdir (pairbin_split_probe.json).

For each build (--lib, one or more library files or source trees with their own build; the first is the reference) and each of --rounds rounds, the builds
alternated, a fresh subprocess with TREEGP_B200_LIB pointing at the build times one TwoD count (CUDA events around
backend.pairbin_packed, L2 overwritten before each, median of 3 after a warm-up) on the bench.py catalogue:
  n1m       N = 1e6, default max_sep (half the field diagonal), unweighted -- the bench value;
  n1m_w     the same, weighted (w uniform in [0.5, 2]);
  cfg4b     N = 1e6 at max_sep = L/100;
  n200k     N = 2e5, default max_sep.
Then, for each build, one profiled count at N = 1e6 (torch.profiler, CUDA activities): kernel time per kernel name,
which separates the classification pass from the pass over the recorded blocks, plus the path fractions.

Prints the card's name, power limit and max SM clock first; they belong beside every number of the record.
Usage: python tools/pairbin_split_probe.py --outdir DIR --lib A.so B.so [--rounds 5]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
    except Exception as e:  # the record still says what it could not read
        out = "unknown (%s)" % e
    return out


def worker(profile):
    import torch

    import bench
    from treegp_b200 import _cabi, backend, binning

    dev = torch.device("cuda", 0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)   # > 126 MB L2
    out = {}

    def catalogue(n, weighted):
        X, y, _, _, mx = bench.make_2pcf_inputs(n)
        px, py = backend.to_device(X[:, 0]), backend.to_device(X[:, 1])
        order = backend.hilbert_order(px, py)
        pk = backend.to_device(y - np.mean(y))[order].contiguous()
        pw = None
        if weighted:
            pw = backend.to_device(np.random.default_rng(7).uniform(0.5, 2.0, n))[order].contiguous()
        off = backend.to_device(np.array([0, n]), torch.int64)
        return px[order].contiguous(), py[order].contiguous(), pk, pw, off, mx

    def count(cat, sep):
        px, py, pk, pw, off, _ = cat
        ed = backend.to_device(binning.twod_thresholds(sep, bench.NBINS))
        return backend.pairbin_packed(px, py, pk, pw, off, int(px.numel()), _cabi.BIN_TWOD, ed, bench.NBINS, 0.0, sep)

    def timed(cat, sep, reps=3):
        count(cat, sep)
        ms = []
        for _ in range(reps):
            flush.fill_(1)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            count(cat, sep)
            b.record()
            torch.cuda.synchronize()
            ms.append(a.elapsed_time(b))
        return float(np.median(ms))

    c1 = catalogue(1_000_000, False)
    out["n1m"] = timed(c1, c1[5])
    out["cfg4b"] = timed(c1, bench.FIELD_2PCF / 100.0)
    cw = catalogue(1_000_000, True)
    out["n1m_w"] = timed(cw, cw[5])
    del cw
    c2 = catalogue(200_000, False)
    out["n200k"] = timed(c2, c2[5])
    if profile:
        from torch.profiler import ProfilerActivity, profile as tprofile

        count(c1, c1[5])
        backend.pairbin_stats(reset=True)
        if hasattr(backend, "pairbin_super_leaves"):
            backend.pairbin_super_leaves(reset=True)
        torch.cuda.synchronize()
        with tprofile(activities=[ProfilerActivity.CUDA]) as prof:
            count(c1, c1[5])
            torch.cuda.synchronize()
        kern = {}
        for ev in prof.key_averages():
            if ev.device_type.name == "CUDA" and "pairbin" in ev.key:
                kern[ev.key] = {"ms": ev.device_time_total / 1e3, "launches": ev.count}
        out["kernels"] = kern
        st = backend.pairbin_stats(reset=True)
        if hasattr(backend, "pairbin_super_leaves"):
            out["super_pairs_leaf_kernel"] = backend.pairbin_super_leaves(reset=True)
        tot = sum(st.values())
        out["path_fractions"] = {k: v / tot for k, v in st.items()} if tot else st
    print("RESULT " + json.dumps(out), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--outdir")
    ap.add_argument("--lib", nargs="+")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--worker", action="store_true")
    ap.add_argument("--profile", action="store_true")
    args = ap.parse_args()
    if args.worker:
        worker(args.profile)
        return
    libs = [os.path.abspath(p) for p in args.lib]

    def run(lib, profile=False):
        # a library file runs under this tree's binding; a directory is a whole tree (binding, library and this
        # probe of its own), for builds whose C ABI differs from this one's
        tree = lib if os.path.isdir(lib) else ROOT
        env = dict(os.environ)
        env.pop("TREEGP_B200_LIB", None)
        if tree == ROOT:
            env["TREEGP_B200_LIB"] = lib
        cmd = [sys.executable, os.path.join(tree, "tools", "pairbin_split_probe.py"), "--worker"] + \
            (["--profile"] if profile else [])
        p = subprocess.run(cmd, env=env, capture_output=True, text=True, cwd=tree)
        for line in p.stdout.splitlines():
            if line.startswith("RESULT "):
                return json.loads(line[7:])
        raise RuntimeError("worker failed (%s):\n%s\n%s" % (lib, p.stdout[-2000:], p.stderr[-4000:]))

    names = {lib: os.path.relpath(lib, ROOT) for lib in libs}   # the record names builds by their place in the tree
    rec = {"card": card(), "libs": [names[lib] for lib in libs], "rounds": []}
    print(rec["card"], flush=True)
    for r in range(args.rounds):
        row = {}
        for lib in (libs if r % 2 == 0 else libs[::-1]):
            row[names[lib]] = run(lib)
            print(r, names[lib], row[names[lib]], flush=True)
        rec["rounds"].append(row)
    rec["profiled"] = {names[lib]: run(lib, profile=True) for lib in libs}
    summary = {}
    for lib in libs:
        s = {}
        for key in ("n1m", "n1m_w", "cfg4b", "n200k"):
            v = np.array([row[names[lib]][key] for row in rec["rounds"]])
            s[key] = {"median_ms": float(np.median(v)), "min_ms": float(v.min()), "max_ms": float(v.max()),
                      "all_ms": v.tolist()}
        summary[names[lib]] = s
    rec["summary"] = summary
    print(json.dumps(summary, indent=1), flush=True)
    if args.outdir:
        os.makedirs(args.outdir, exist_ok=True)
        with open(os.path.join(args.outdir, "pairbin_split_probe.json"), "w") as f:
            json.dump(rec, f)


if __name__ == "__main__":
    main()
