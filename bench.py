#!/usr/bin/env python
"""bench.py -- headline measurement of the treegp_b200 hot path.

BASELINE.json metric: "GP fit+predict wall-s at N=40k; 2PCF pairs/s at 1/2/4/8 B200".

One JSON line is printed (rank 0).  Its primary metric is the one that is defined at 1/2/4/8 GPUs:

  metric  = "2pcf_pairs_per_s": unordered pairs binned per second by the anisotropic TwoD pair-binning
            kernel on N = 1,000,000 synthetic points (configs[3]; nbins = 21, min_sep = 0, max_sep = the
            reference default: half the field diagonal, two_pcf.py:421 -> 84 % of all pairs land in a bin).
            A "step" is one complete pair count over all N(N-1)/2 pairs.  With --gpus N the pair tiles are
            dealt to the ranks and the bin sums all-reduced over NCCL: total work is fixed -> "strong".
  e2e     = the same count through the reference-facing API, treegp_b200.two_pcf(...).comp_2pcf(X, y,
            y_err) with HOST numpy inputs (H2D of the points and D2H of xi inside the timed region).
  gp      = the other half of the BASELINE metric (configs[2]): wall seconds of GPInterpolation.initialize +
            solve(optimizer='anisotropic') + predict(1e6 points) for a 2-D AnisotropicVonKarman field with
            N = 40,000; the diagonal predictive variance for ALL 1e6 points (sharded over the ranks), the full
            covariance of a 4096-point subset, kernel-level rooflines.  Short numbers under "gp", details under
            "gp_fit_predict".
  cfg     = the remaining BASELINE.json configs: cfg2 (N = 10k log-likelihood fit; with --gpus N the
            forward-difference probes of every L-BFGS-B gradient are dealt to the ranks), cfg4b (the 2PCF at
            max_sep = L/100), cfg5 (N = 200k: meanify + KNN mean subtraction + 100 bootstrap resamples + robust fit).
  cpu_baseline = the CPU restatements (oracle/) timed on this box's host cores on bounded samples: the pair binning
            (OpenMP C) and the GP pieces (numpy/scipy, as the reference computes them) with the N^2 / N^3
            extrapolation to configs[2] stated.  Rank 0, --gpus 1 only.

`--impl reference` times the same CPU restatements alone (TreeCorr itself is not installable here).
`--dump-outputs DIR` saves the bin sums of the last timed pair count (DIR/npairs.npy, sumw.npy, sumwkk.npy).
"""
import argparse
import json
import os
import re
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--npoints", type=int, default=1_000_000, help="2PCF points (configs[3]: 1e6)")
    ap.add_argument("--gp-train", type=int, default=40_000, help="GP training points (configs[2]: 40k)")
    ap.add_argument("--gp-predict", type=int, default=1_000_000)
    ap.add_argument("--var-points", type=int, default=-1, help="test points of the diagonal-variance run (-1: all)")
    ap.add_argument("--skip-gp", action="store_true", help="only the 2PCF part (used for ncu captures)")
    ap.add_argument("--skip-var", action="store_true", help="skip the all-M diagonal variance (N^2 M flop)")
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--skip-other", action="store_true", help="skip the cfg2 / cfg4b / cfg5 side measurements")
    ap.add_argument("--cpu-rows", type=int, default=20000, help="rows of the pair matrix in the CPU sample")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the bin sums of the last timed 2PCF step as DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    return args


# ------------------------------------------------------------------------------------------------
# synthetic inputs (SURVEY.md section 8d)
# ------------------------------------------------------------------------------------------------
FIELD_2PCF = 1000.0
NBINS = 21


def make_2pcf_inputs(n, seed=42):
    rng = np.random.default_rng(seed)
    X = rng.uniform(-FIELD_2PCF / 2, FIELD_2PCF / 2, size=(n, 2))
    y = rng.normal(size=n)  # pair counts and timing do not depend on the field values
    y_err = np.zeros(n)
    max_sep = np.sqrt(2.0) * FIELD_2PCF / 2.0  # reference default: half the field diagonal
    return X, y, y_err, 0.0, max_sep


def gp_problem(n, m):
    """configs[2]: coordinates, kernel string and its parameters (the field values are drawn on the device)."""
    from treegp_b200.two_pcf import get_correlation_length_matrix

    L = 160.0 * np.sqrt(n / 40000.0)
    size, g1, g2, sigma, noise = 1.5, 0.2, 0.2, 2.0, 0.01
    inv = np.linalg.inv(get_correlation_length_matrix(size, g1, g2))
    kstr = "%r**2 * AnisotropicVonKarman(invLam=array([[%.17g, %.17g], [%.17g, %.17g]]))" % (
        sigma, inv[0, 0], inv[0, 1], inv[1, 0], inv[1, 1])
    rng = np.random.default_rng(42)
    X = rng.uniform(-L / 2, L / 2, size=(n, 2))
    Xs = rng.uniform(-L / 2, L / 2, size=(m, 2))
    return X, Xs, kstr, inv, sigma, noise, rng


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    def __init__(self, index=0):
        super().__init__(daemon=True)
        self.index = index
        self.rows = []
        self._stop_evt = threading.Event()

    def run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        # one nvidia-smi process sampling every 50 ms (a fresh process per sample takes ~0.2 s to start, which is
        # as long as a whole timed step by now)
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return
        for line in self.proc.stdout:
            parts = [p.strip() for p in line.strip().split(",")]
            if len(parts) >= 7:
                self.rows.append(parts)
            if self._stop_evt.is_set():
                break

    def stop(self):
        self._stop_evt.set()
        if getattr(self, "proc", None) is not None:
            try:
                self.proc.terminate()
            except Exception:
                pass
        self.join(timeout=3)
        sm = [float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[3 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(self.rows)}


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            d = json.load(fh)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


_UNIT = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9, "Tbyte": 1e12}


def ncu_summary(name):
    """Numbers of a committed ncu summary (profiles/<name>, written by tools/ncu_summary.py from an
    `ncu --set full` capture): DRAM traffic per launch and what bounds the kernel.  None if the file is absent."""
    path = os.path.join(ROOT, "profiles", name)
    if not os.path.exists(path):
        return None
    vals = {}
    with open(path) as fh:
        for ln in fh:
            m = re.match(r"^(\S+)\s+(\S+)?\s+([-0-9.eE+]+)\s*$", ln)
            if m:
                vals[m.group(1)] = (m.group(2) or "", float(m.group(3)))

    def get(key, scale_units=False):
        if key not in vals:
            return None
        unit, v = vals[key]
        return v * _UNIT.get(unit, 1.0) if scale_units else v

    rd, wr = get("dram__bytes_read.sum", True), get("dram__bytes_write.sum", True)
    return {"source": "profiles/" + name,
            "traffic": None if rd is None or wr is None else rd + wr,
            "issue_active_pct": get("smsp__issue_active.avg.pct_of_peak_sustained_active"),
            "warps_active_pct": get("sm__warps_active.avg.pct_of_peak_sustained_active"),
            "fp64_pipe_pct": get("sm__pipe_fp64_cycles_active.avg.pct_of_peak_sustained_active"),
            "no_instruction_stall_per_issue": get("smsp__average_warps_issue_stalled_no_instruction_per_issue_active.ratio"),
            "registers": get("launch__registers_per_thread")}


# ------------------------------------------------------------------------------------------------
# CPU baselines / reference arm
# ------------------------------------------------------------------------------------------------
def _all_host_threads():
    # torchrun exports OMP_NUM_THREADS=1 to every rank; the CPU baseline is meant to use all host cores
    if int(os.environ.get("WORLD_SIZE", "1")) > 1 or "OMP_NUM_THREADS" not in os.environ:
        os.environ["OMP_NUM_THREADS"] = str(os.cpu_count())


def cpu_pairbin_sample(X, y, min_sep, max_sep, rows):
    """Time the oracle (C, OpenMP, all host cores) on rows [0, rows) of the pair matrix."""
    _all_host_threads()
    from oracle import pairbin_oracle as po

    if int(os.environ.get("WORLD_SIZE", "1")) > 1:
        po.set_threads(os.cpu_count())  # the OpenMP runtime may already be initialised with 1 thread
    n = len(y)
    rows = min(rows, n)
    k = y - np.mean(y)
    t0 = time.perf_counter()
    po.pairbin(X[:, 0], X[:, 1], k, None, min_sep, max_sep, NBINS, "TwoD", rows=(0, rows))
    dt = time.perf_counter() - t0
    pairs = rows * n - rows * (rows + 1) // 2
    return pairs / dt, dt, pairs, po.num_threads()


def cpu_gp_sample(n_target, m_target, nk=3000, nc=6000, mp_=1500):
    """The GP half of the metric on the host cores, as the reference computes it (oracle/gp_oracle.py: numpy / scipy
    restatement of kernels.py:359-381, log_likelihood.py:29-37, gp_interp.py:177-183, pinned to the reference by
    tests/test_oracle_golden.py), on bounded sizes, with the N^2 / N^3 / M N extrapolation to configs[2]."""
    _all_host_threads()
    from oracle import gp_oracle as go
    from scipy.linalg import cho_solve, cholesky

    X, Xs, kstr, inv, sigma, noise, rng = gp_problem(n_target, 4 * mp_)
    amp = sigma ** 2
    t0 = time.perf_counter()
    K = go.kmat("vonkarman", X[:nk], amp=amp, invLam=inv)
    t_k = time.perf_counter() - t0
    t0 = time.perf_counter()
    Ks = go.kmat("vonkarman", Xs[:mp_], X[:nk], amp=amp, invLam=inv)
    t_ks = time.perf_counter() - t0
    del K, Ks
    # Cholesky + solve on a well-conditioned RBF matrix of size nc (the arithmetic does not depend on the kernel)
    Kc = go.kmat("rbf", X[:nc] * 4.0, amp=amp, invLam=inv) + np.eye(nc) * 0.5
    yv = rng.normal(size=nc)
    t0 = time.perf_counter()
    U = cholesky(Kc, lower=False)
    t_chol = time.perf_counter() - t0
    t0 = time.perf_counter()
    alpha = cho_solve((U, False), yv)
    t_solve = time.perf_counter() - t0
    t0 = time.perf_counter()
    _ = np.ones((mp_, nc)) @ alpha
    t_mv = time.perf_counter() - t0
    ex = {"kmat_s": t_k * (n_target / nk) ** 2, "potrf_s": t_chol * (n_target / nc) ** 3,
          "potrs_s": t_solve * (n_target / nc) ** 2,
          "predict_mean_s": (t_ks / (mp_ * nk) + t_mv / (mp_ * nc)) * m_target * n_target}
    return {"kind": "port", "cores": os.cpu_count(), "unit": "s",
            "value": float(sum(ex.values())),
            "sample": "K(X,X) von Karman at N=%d: %.2f s; K(X*,X) %dx%d: %.2f s; cholesky at N=%d: %.2f s (%.0f GFLOP/s); "
                      "cho_solve: %.3f s" % (nk, t_k, mp_, nk, t_ks, nc, t_chol, nc ** 3 / 3 / t_chol / 1e9, t_solve),
            "extrapolated_to_N=%d_M=%d_s" % (n_target, m_target): {k: float(v) for k, v in ex.items()},
            "extrapolation": "K build ~ N^2, Cholesky ~ N^3, solve ~ N^2, predict ~ M N (K* is built in row chunks; "
                             "scipy.special.kv is single-threaded, the BLAS calls use all cores)",
            "note": "oracle/gp_oracle.py = numpy/scipy restatement of the reference (pinned to it by golden vectors); "
                    "one fit evaluation + predict mean, no optimiser loop, no variance"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    X, y, y_err, mn, mx = make_2pcf_inputs(args.npoints)
    rates = []
    for i in range(args.warmup + args.steps):
        rate, dt, pairs, cores = cpu_pairbin_sample(X, y, mn, mx, args.cpu_rows)
        if i >= args.warmup:
            rates.append((rate, dt))
    value = float(np.mean([r for r, _ in rates]))
    ms = float(np.mean([d for _, d in rates]) * 1e3)
    sample = "rows [0,%d) of the N=%d pair matrix = %.3g unordered pairs per step" % (args.cpu_rows, args.npoints, pairs)
    line = {
        "impl": "reference", "metric": "2pcf_pairs_per_s", "value": value, "unit": "pairs/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "anisotropic TwoD 2PCF pair binning, N=%d, nbins=21, min_sep=0, max_sep=half field "
                               "diagonal (configs[3])" % args.npoints},
        "cpu_baseline": {"value": value, "unit": "pairs/s", "cores": cores, "kind": "port", "sample": sample,
                         "note": "oracle/pairbin_oracle.c: O(N^2) brute-force CPU port (OpenMP); NOT TreeCorr (not "
                                 "installable), whose bin_slop=0 tree traversal visits fewer than N^2/2 pairs"},
        "e2e": {"value": value, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    if not args.skip_gp:
        line["gp_fit_predict"] = {"metric": "gp_fit_predict_wall_s", "cpu_baseline": cpu_gp_sample(args.gp_train, args.gp_predict)}
        line["gp"] = {"cpu_extrapolated_wall_s": line["gp_fit_predict"]["cpu_baseline"]["value"]}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as tdist

    import treegp_b200 as treegp
    from treegp_b200 import _cabi, backend, binning, dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        tdist.init_process_group("nccl", device_id=dev)
    _cabi.load()

    def barrier():
        if world > 1:
            tdist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        tdist.all_reduce(t, op=tdist.ReduceOp.MAX)
        return float(t.item())

    ctx = dict(rank=rank, world=world, dev=dev, barrier=barrier, max_over_ranks=max_over_ranks, tdist=tdist)
    hbm_peak, peak_src = load_peaks()
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2

    # ---------------- 2PCF: device-resident timing ----------------
    n = args.npoints
    X, y, y_err, mn, mx = make_2pcf_inputs(n)
    npairs_total = n * (n - 1) // 2
    px, py = backend.to_device(X[:, 0]), backend.to_device(X[:, 1])
    pk = backend.to_device(y - np.mean(y))
    # device-resident inputs are stored in Hilbert order (what two_pcf.comp_2pcf does on the way in)
    order = backend.hilbert_order(px, py)
    px, py, pk = px[order].contiguous(), py[order].contiguous(), pk[order].contiguous()
    off = backend.to_device(np.array([0, n]), torch.int64)
    edges = backend.to_device(binning.twod_thresholds(mx, NBINS))
    launches = 0
    # the exchange step behind the C ABI (tgp_allreduce_bins: NCCL bound by the library at run time); torch.distributed's
    # all-reduce if that communicator cannot be made
    comm, collective = None, "none"
    if world > 1:
        try:
            comm = dist.CabiComm(rank, world)
            collective = "tgp_allreduce_bins (C ABI, NCCL via dlopen)"
        except Exception as exc:      # noqa: BLE001
            collective = "torch.distributed all_reduce (CabiComm failed: %s)" % (exc,)

    def reduce_bins(res):
        if comm is not None:
            return comm.allreduce_packed_bins(res)          # plane 0 stays int64 words
        return dist.allreduce_packed_bins(dist.WORLD, res)  # plane 0 becomes FP64 values

    counts_are_words = world == 1 or comm is not None

    def count(sep, ed):
        """one device-resident step: pair count of this rank's tiles (+ ONE all-reduce of the packed bin sums)"""
        res = backend.pairbin_packed(px, py, pk, None, off, n, _cabi.BIN_TWOD, ed, NBINS, mn, sep, rank=rank, nranks=world)
        return res

    def timed_counts(sep, ed, reps):
        step_ms, kern_ms = [], []
        res = None
        for _ in range(reps):
            flush_buf.fill_(1)
            barrier()
            e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
            e0.record()
            res = count(sep, ed)
            e1.record()
            if world > 1:
                res = reduce_bins(res)
            e2.record()
            barrier()
            step_ms.append(max_over_ranks(e0.elapsed_time(e2)))
            kern_ms.append(max_over_ranks(e0.elapsed_time(e1)))
        return res, step_ms, kern_ms

    def total_count(res):
        return int(res[0].view(torch.int64).sum().item()) if counts_are_words else int(res[0].sum().item())

    # per-pair mode first (block forms off: every pair of every in-range block goes through the compare /
    # masked-FMA loop): this is the kernel the FP64-issue roofline of 10 ops per pair applies to
    backend.set_option("pairbin_block_sums", 0)
    count(mx, edges)
    res_pp, _, pp_ms = timed_counts(mx, edges, 2)
    backend.set_option("pairbin_block_sums", 1)
    backend.pairbin_stats(reset=True)

    for _ in range(args.warmup):
        res = count(mx, edges)
    barrier()
    stats = backend.pairbin_stats(reset=True)   # paths taken by one rank's share during the warm-up steps
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    res, step_ms, kern_ms = timed_counts(mx, edges, args.steps)
    launches += 2 * args.steps  # pairbin_boxes_kernel + pairbin_kernel (ours); the counter memset and torch fills are not counted
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_pairbin(args.dump_outputs, res.cpu().numpy(), counts_are_words)
    counted = total_count(res)
    total_ms = float(np.sum(step_ms))
    value = npairs_total * args.steps / (total_ms * 1e-3)
    as_int = (lambda t: t[0].view(torch.int64)) if counts_are_words else (lambda t: t[0])
    same_counts = bool(total_count(res_pp) == counted and torch.equal(as_int(res_pp), as_int(res)))

    # ---------------- 2PCF: end to end through the public API (host buffers) ----------------
    def pinned(a):
        """numpy view of a page-locked copy of `a` (the contract's "inputs from pinned host memory"): the API
        takes plain numpy arrays; the driver recognises the pages as pinned and copies them by DMA"""
        t = torch.empty(a.shape, dtype=torch.float64, pin_memory=True)
        v = t.numpy()      # keeps `t` alive as its base
        v[...] = a
        return v

    Xp, yp, yerrp = pinned(np.ascontiguousarray(X)), pinned(y), pinned(y_err)
    e2e_ms = []
    tp = treegp.two_pcf(Xp, yp, yerrp, mn, mx, nbins=NBINS, anisotropic=True)
    tp.group = (comm if comm is not None else dist.WORLD) if world > 1 else False
    for i in range(2 + args.steps):
        barrier()
        t0 = time.perf_counter()
        xi, _, _, _ = tp.comp_2pcf(Xp, yp, yerrp)
        torch.cuda.synchronize()
        dt = max_over_ranks((time.perf_counter() - t0) * 1e3)
        if i > 1:
            e2e_ms.append(dt)
    e2e_value = npairs_total / (float(np.mean(e2e_ms)) * 1e-3)
    h2d = 3 * 8 * n + 8 * (NBINS + 1) + 16
    d2h = NBINS * NBINS * (8 + 8 + 8)

    # ---------------- FP64 peaks (roofline denominators), measured live ----------------
    dfma_tf = backend.microbench_fp64(0, 20000)
    dmma_tf = backend.microbench_fp64(1, 20000)
    # algorithmic work per unordered pair: 10 FP64 operations (SURVEY.md section 8d); peak in operations/s is
    # the measured DFMA rate / 2 (one FMA instruction = 2 flop = 1 operation slot)
    ops_per_pair = 10.0
    my_pairs = npairs_total / world
    peak_gops = dfma_tf * 1e3 / 2.0
    kern_s = float(np.mean(kern_ms)) * 1e-3
    pp_s = float(np.mean(pp_ms)) * 1e-3
    st_tot = max(1, sum(stats.values()))
    frac_paths = {k: v / st_tot for k, v in stats.items()}
    ach_pp = ops_per_pair * my_pairs / pp_s / 1e9
    ncu_w = ncu_summary("r2_pairbin_witness_N1M.ncu.txt") if (n == 1_000_000 and world == 1) else None
    ncu_t = ncu_summary("r2_pairbin_timed_N1M.ncu.txt") if (n == 1_000_000 and world == 1) else None
    roofline = {
        "bound": "fp64_alu", "kernel": "pairbin_kernel<TwoD, unweighted, pair-by-pair> (witness: the instantiation the "
                                       "10-ops-per-pair figure describes)",
        "achieved": ach_pp, "peak": peak_gops, "unit": "Gop/s (FP64 instructions x lanes)", "frac": ach_pp / peak_gops,
        "traffic": None if ncu_w is None else ncu_w["traffic"],
        "traffic_source": None if ncu_w is None else ncu_w["source"],
        "ms_per_launch": pp_s * 1e3, "pairs_per_s": my_pairs * world / pp_s,
        # what bounds the SHIPPED (timed) kernel: it does less than brute-force work, so the algorithmic
        # 10 ops/pair figure over its time exceeds the FP64 peak (algorithmic_frac > 1 is not a typo)
        "timed": {"kernel": "pairbin_kernel<TwoD, unweighted, block forms> (value / ms_per_step)",
                  "ms_per_launch": kern_s * 1e3, "algorithmic_frac": ops_per_pair * my_pairs / kern_s / 1e9 / peak_gops,
                  "speedup_over_witness": pp_s / kern_s, "counts_identical_to_witness": same_counts,
                  "path_fractions": frac_paths,
                  "traffic": None if ncu_t is None else ncu_t["traffic"],
                  "algorithmic_bytes": 24.0 * n,
                  "issue_active_pct": None if ncu_t is None else ncu_t["issue_active_pct"],
                  "warps_active_pct": None if ncu_t is None else ncu_t["warps_active_pct"],
                  "no_instruction_stall_per_issue": None if ncu_t is None else ncu_t["no_instruction_stall_per_issue"],
                  "ncu_source": None if ncu_t is None else ncu_t["source"]},
        "hbm_GBs_of_timed_kernel": 24.0 * n / kern_s / 1e9, "hbm_peak_GBs": hbm_peak, "hbm_peak_source": peak_src}

    line = {
        "metric": "2pcf_pairs_per_s", "value": value, "unit": "pairs/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "anisotropic TwoD 2PCF pair binning, N=%d, nbins=21, min_sep=0, max_sep=half field "
                               "diagonal (configs[3])" % n,
                   "pairs_per_step": npairs_total, "pairs_in_range_x2": counted,
                   "sharding": "pair tiles over %d rank(s) + ONE NCCL allreduce of the packed bin sums" % world,
                   "collective": collective,
                   "l2": "256 MB buffer written between timed iterations (L2 flush)"},
        "e2e": {"value": e2e_value, "unit": "pairs/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_call": float(np.mean(e2e_ms)),
                "collective": collective,
                "api": "treegp_b200.two_pcf(...).comp_2pcf(X, y, y_err) with host numpy inputs (page-locked)"},
        "gpu_launches": launches,
        "clocks": clocks,
        "gp": None, "cfg": None,          # short numbers, filled below (kept early in the line on purpose)
        "roofline": roofline,
        "fp64_peaks_measured": {"dfma_tflops": dfma_tf, "dmma_tflops": dmma_tf},
    }

    # ---------------- cfg4b: the same catalogue at max_sep = L/100 (0.1 % of the pairs in range) ----------------
    cfg = {}
    if not args.skip_other:
        sep_b = FIELD_2PCF / 100.0
        edges_b = backend.to_device(binning.twod_thresholds(sep_b, NBINS))
        count(sep_b, edges_b)
        res_b, step_b, _ = timed_counts(sep_b, edges_b, 3)
        cfg["cfg4b_pairs_per_s"] = npairs_total / (float(np.mean(step_b)) * 1e-3)
        cfg["cfg4b_ms"] = float(np.mean(step_b))
        cfg["cfg4b_in_range_frac"] = total_count(res_b) / 2.0 / npairs_total
    del px, py, pk, flush_buf
    torch.cuda.empty_cache()

    # ---------------- GP fit + predict at N = 40k ----------------
    if not args.skip_gp:
        gp_short, gp_long = run_gp(args, treegp, backend, dist, ctx, hbm_peak, dmma_tf)
        line["gp"] = gp_short
        line["gp_fit_predict"] = gp_long
    if not args.skip_other:
        cfg.update(run_cfg2(args, treegp, backend, ctx))
        if world == 1:
            cfg.update(run_cfg5(args, treegp, backend, ctx))
        else:
            cfg.update(run_bootstrap_sharded(args, treegp, backend, dist, ctx))
    line["cfg"] = cfg or None

    # ---------------- CPU baselines (rank 0, one GPU, bounded samples) ----------------
    if rank == 0 and world == 1 and not args.skip_cpu:
        rate, dt, pairs, cores = cpu_pairbin_sample(X, y, mn, mx, args.cpu_rows)
        line["cpu_baseline"] = {"value": rate, "unit": "pairs/s", "cores": cores, "kind": "port",
                                "sample": "rows [0,%d) of the N=%d pair matrix = %.3g unordered pairs, %.1f s"
                                          % (args.cpu_rows, n, pairs, dt),
                                "note": "oracle/pairbin_oracle.c: O(N^2) brute-force CPU port (OpenMP); NOT TreeCorr (not "
                                        "installable), whose bin_slop=0 tree traversal visits fewer than N^2/2 pairs"}
        if not args.skip_gp:
            cg = cpu_gp_sample(args.gp_train, args.gp_predict)
            line["gp_fit_predict"]["cpu_baseline"] = cg
            line["gp"]["cpu_extrapolated_wall_s"] = cg["value"]
    line["notes"] = {
        "roofline": "neither HBM- nor tensor-bound: 24 N bytes in, N^2/2 pairs; peak = measured DFMA issue rate "
                    "(tgp_microbench_fp64); algorithmic work 10 FP64 ops per unordered pair (SURVEY 8d).  achieved / frac "
                    "are measured live on the pair-by-pair instantiation (block forms off).  The TIMED kernel books blocks "
                    "of 32 x 32 pairs that provably fall into one bin from chunk sums, answers one-axis blocks by a rank "
                    "query on sorted chunks and 2 x 2-window blocks from two such queries: identical counts "
                    "(roofline.timed); traffic / issue-active / warps-active are read from the committed ncu summaries.",
        "vs_reference": "the reference arm is an O(N^2) CPU port on a row sample, not TreeCorr: its ratio is a stated "
                        "baseline, not a speed-up over treegp",
        "gp": "gp.wall_s is the public GPInterpolation path, which factorises K inside its envelope when the kernel's "
              "support (correlation >= 1e-40 amp) is short against the field (points sorted along one axis; "
              "gp.potrf_envelope_s, flops = gp.potrf_envelope_flops_frac of N^3/3; same logL / alpha / mean to "
              "rounding, tests/test_gpu_envelope.py).  gp.potrf_s / potrf_tflops / potrf_frac_dmma are the DENSE "
              "factorisation of the same matrix (what the reference's scipy call and cuSOLVER do), kept as the "
              "tensor-pipe roofline figure.  gp.var_all_M_s uses windows + envelopes (gp_fit_predict.variance.*plan), "
              "gp.var_plain_* are the plain solves on the cached factor, timed on a subset and extrapolated.",
    }
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        tdist.destroy_process_group()


def dump_pairbin(out_dir, host, counts_are_words):
    """What backend.pairbin returns for the last timed step -- pair counts, sum w and sum w k k, each shaped
    (catalogues, NBINS * NBINS) -- as float64 .npy files.  The inputs are seeded, so two builds run with the same
    arguments can be compared output for output: the counts and sum w exactly, sum w k k to rounding (the kernel
    accumulates it with FP64 atomics, whose order varies from run to run)."""
    os.makedirs(out_dir, exist_ok=True)
    counts = np.ascontiguousarray(host[0]).view(np.int64) if counts_are_words else host[0]
    for name, a in (("npairs", counts), ("sumw", host[1]), ("sumwkk", host[2])):
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float64))


def _ev(torch, fn, reps=2):
    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b) * 1e-3)
    return float(np.mean(ts))


def run_gp(args, treegp, backend, dist, ctx, hbm_peak, dmma_tf):
    """configs[2]: 2-D AnisotropicVonKarman, N train / M predict, optimizer='anisotropic'."""
    import torch
    from treegp_b200.kernels import lower_kernel

    rank, world, dev, barrier, max_over_ranks = (ctx[k] for k in ("rank", "world", "dev", "barrier", "max_over_ranks"))
    n, m = args.gp_train, args.gp_predict
    X, Xs, kstr, inv, sigma, noise, rng = gp_problem(n, m)
    kern = treegp.eval_kernel(kstr)
    # exact GRF draw y = L z + noise with the library's own K build + Cholesky (data generation, not timed)
    y, y_err = treegp.sample_grf(kern, X, noise=noise, seed=43)
    torch.cuda.empty_cache()

    lo, hi = dist.slab(m, rank, world)
    Xs_local = Xs[lo:hi]

    def one_run():
        t = {}
        barrier()
        t0 = time.perf_counter()
        gp = treegp.GPInterpolation(kernel=kstr, optimizer="anisotropic", normalize=True, nbins=21, min_sep=0.0,
                                    max_sep=1.0, p0=[1.0, 0.0, 0.0])
        gp.initialize(X, y, y_err=y_err)
        gp.solve()
        torch.cuda.synchronize()
        t["solve_anisotropic_s"] = time.perf_counter() - t0
        t1 = time.perf_counter()
        ypred = gp.predict(Xs_local)
        if world > 1:  # every rank ends up with all M predictions (all-gather of the slabs, 8 M bytes)
            ypred = dist.gather_slabs(torch.as_tensor(ypred, device=dev), m).cpu().numpy()
        torch.cuda.synchronize()
        t["predict_s"] = time.perf_counter() - t1
        t["total_s"] = time.perf_counter() - t0
        return gp, ypred, t

    one_run()  # warm-up (allocator, kernel load)
    runs = []
    for _ in range(2):
        gp, ypred, t = one_run()
        runs.append({k: max_over_ranks(v) for k, v in t.items()})
    best = min(runs, key=lambda r: r["total_s"])

    # ---- cfg3 as written: diagonal variance for ALL M test points (sharded), full covariance of a 4096 subset ----
    var = {}
    if not args.skip_var:
        mv = len(Xs_local) if args.var_points < 0 else min(len(Xs_local), max(1, args.var_points // world))
        barrier()
        t0 = time.perf_counter()
        _, v_local = gp.predict_var(Xs_local[:mv])
        torch.cuda.synchronize()
        t_var = max_over_ranks(time.perf_counter() - t0)
        plan = dict(getattr(gp, "_var_plan", {}) or {})
        done_flops = (plan["flops_windowed"] + plan["flops_factors"]) if plan.get("used") else float(n) * n * mv
        var = {"predict_var_diag_points_total": mv * world, "predict_var_diag_s": t_var,
               # flops actually executed (trailing sub-systems + the two extra factorisations when windowed)
               "predict_var_diag_tflops_per_gpu": done_flops / t_var / 1e12,
               "predict_var_diag_plain_equivalent_tflops_per_gpu": float(n) * n * mv / t_var / 1e12,
               "predict_var_windowed": bool(plan.get("used", False)), "predict_var_plan": plan,
               "var_min": float(np.min(v_local)), "var_max": float(np.max(v_local))}
        # the plain solves on the cached (unsorted) factor, on a bounded subset: time per point and agreement
        mp = min(mv, 2 * backend.var_chunk(n, mv))
        gp.WINDOWED_VARIANCE = False
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        _, v_plain = gp.predict_var(Xs_local[:mp])
        torch.cuda.synchronize()
        t_plain = time.perf_counter() - t0
        gp.WINDOWED_VARIANCE = True
        var["predict_var_plain_subset_points"] = mp
        var["predict_var_plain_subset_s"] = t_plain
        var["predict_var_plain_extrapolated_all_points_s"] = t_plain * mv / mp
        var["predict_var_plain_tflops_per_gpu"] = float(n) * n * mp / t_plain / 1e12
        var["windowed_minus_plain_max"] = float(np.max(np.abs(v_plain - v_local[:mp])))
        if rank == 0:
            mc = min(4096, len(Xs_local))
            gp.predict(Xs_local[:64], return_cov=True)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            _, cov = gp.predict(Xs_local[:mc], return_cov=True)
            torch.cuda.synchronize()
            var["predict_full_cov_M=%d_s" % mc] = time.perf_counter() - t0
            # the diagonal of the full covariance is the diagonal variance
            var["cov_diag_minus_var_max"] = float(np.max(np.abs(np.diag(cov) - v_local[:mc])))
        barrier()

    # ---- kernel-level breakdown with CUDA events (device-resident, rank-local) ----
    ev = lambda fn, reps=2: _ev(torch, fn, reps)
    desc = lower_kernel(gp.kernel, 2)
    gp._alpha = gp._factor = gp._alpha_dev = None
    del gp
    torch.cuda.empty_cache()
    Xd = backend.as_points(X)
    e2 = backend.to_device(y_err ** 2)
    ws = backend.alloc_matrix(n, n)
    t_k = ev(lambda: backend.kmat_sym(Xd, desc, e2, out=ws, lower_only=True))

    def build_and_factor():
        backend.kmat_sym(Xd, desc, e2, out=ws, lower_only=True)
        backend.potrf(ws, n)

    # the same build for an RBF metric, full square as kernel.__call__(X) returns it: the HBM-store-bound case
    desc_rbf = lower_kernel(treegp.eval_kernel(kstr.replace("AnisotropicVonKarman", "AnisotropicRBF")), 2)
    t_k_rbf_full = ev(lambda: backend.kmat_sym(Xd, desc_rbf, e2, out=ws, lower_only=False), reps=3)
    t_kf = ev(build_and_factor)
    t_chol = t_kf - t_k
    # the factorisation GPInterpolation runs for this kernel: inside the envelope of K (points sorted along one axis)
    env = backend.plan_envelope(Xd, desc)
    t_chol_env = None
    if env is not None:
        Xo, e2o = Xd[env["order"]].contiguous(), e2[env["order"]].contiguous()

        def build_and_factor_env():
            backend.kmat_sym(Xo, desc, e2o, out=ws, lower_only=True)
            backend.potrf(ws, n, row_end=env["row_end"])

        t_chol_env = ev(build_and_factor_env) - t_k
        del Xo, e2o
    # cuSOLVER's Dpotrf on the same matrix (torch.linalg.cholesky), for comparison only
    t_cusolver = None
    try:
        backend.kmat_sym(Xd, desc, e2, out=ws, lower_only=False)
        Kfull = ws[:, :n]
        t_cusolver = ev(lambda: torch.linalg.cholesky(Kfull), reps=1)
        del Kfull
    except Exception:
        pass
    build_and_factor()
    b = backend.to_device(y)
    t_solve = ev(lambda: backend.potrs_vec(ws, n, b.clone()), reps=3)
    Xsd = backend.as_points(Xs_local)
    alpha = backend.potrs_vec(ws, n, b.clone())
    t_mean_full = ev(lambda: backend.predict_mean(Xsd, Xd, desc, alpha, truncate=False))
    t_mean = ev(lambda: backend.predict_mean(Xsd, Xd, desc, alpha))   # what predict() runs: truncated support
    flops = n ** 3 / 3.0
    short = {"wall_s": best["total_s"], "solve_s": best["solve_anisotropic_s"], "predict_s": best["predict_s"],
             "potrf_s": t_chol, "potrf_tflops": flops / t_chol / 1e12, "potrf_frac_dmma": flops / t_chol / 1e12 / dmma_tf,
             "cusolver_potrf_s": t_cusolver,
             "potrf_envelope_s": t_chol_env,
             "potrf_envelope_flops_frac": None if env is None else env["flops"] / env["flops_dense"],
             "potrs_vec_s": t_solve, "potrs_GBs": 8.0 * n * n / t_solve / 1e9,
             "potrs_frac_hbm": 8.0 * n * n / t_solve / 1e9 / hbm_peak,
             "kmat_rbf_frac_hbm": 8.0 * n * n / t_k_rbf_full / 1e9 / hbm_peak,
             "var_all_M_s": var.get("predict_var_diag_s"), "var_tflops_per_gpu": var.get("predict_var_diag_tflops_per_gpu"),
             "var_points": var.get("predict_var_diag_points_total"), "var_windowed": var.get("predict_var_windowed"),
             "var_plain_all_M_s": var.get("predict_var_plain_extrapolated_all_points_s"),
             "var_plain_tflops_per_gpu": var.get("predict_var_plain_tflops_per_gpu"),
             "var_windowed_minus_plain_max": var.get("windowed_minus_plain_max")}
    long = {
        "metric": "gp_fit_predict_wall_s", "value": best["total_s"], "unit": "s", "higher_is_better": False,
        "config": {"workload": "2D AnisotropicVonKarman GP, N=%d train / M=%d predict (configs[2]); "
                               "GPInterpolation.initialize + solve(optimizer='anisotropic', nbins=21, max_sep=1 as tests/test_hyp_search.py, 444 bootstraps) "
                               "+ predict(M), host numpy in/out; test points sharded over %d rank(s)" % (n, m, world)},
        "wall_breakdown_s": best,
        "kernel_breakdown_s": {"kmat_lower": t_k, "kmat_rbf_full": t_k_rbf_full, "potrf": t_chol, "potrs_vec": t_solve,
                               "cusolver_potrf": t_cusolver,
                               "predict_mean_local_M=%d" % len(Xs_local): t_mean,
                               "predict_mean_full_sum_local_M=%d" % len(Xs_local): t_mean_full},
        "variance": var,
        "fitted_theta": [float(v) for v in desc_theta(treegp, desc, kern)],
        "true_theta": [float(v) for v in kern.theta],
        "roofline_potrf": {"bound": "tensor", "kernel": "gemm_nt_sub_kernel (DMMA.8x8x4) inside tgp_potrf",
                           "achieved": flops / t_chol / 1e12, "peak": dmma_tf, "unit": "TFLOP/s",
                           "frac": flops / t_chol / 1e12 / dmma_tf,
                           "note": "FP64 tensor pipe (mma.sync m8n8k4 f64); peak measured live by tgp_microbench_fp64"},
        "roofline_kmat": {"bound": "hbm", "kernel": "kmat_sym_kernel<RBF>, full N x N", "achieved": 8.0 * n * n / t_k_rbf_full / 1e9,
                          "peak": hbm_peak, "unit": "GB/s", "frac": 8.0 * n * n / t_k_rbf_full / 1e9 / hbm_peak,
                          "note": "AnisotropicRBF, full square (what kernel.__call__(X) returns), algorithmic bytes 8 N^2 "
                                  "stored once; the von Karman build of this fit (kmat_lower above, 4 N^2 bytes) is "
                                  "FP64-ALU bound by the Bessel-K evaluation",
                          "von_karman_lower_GBs": 4.0 * n * n / t_k / 1e9},
        "roofline_potrs": {"bound": "hbm", "kernel": "triangular sweeps (tgp_potrs_vec)", "achieved": 8.0 * n * n / t_solve / 1e9,
                           "peak": hbm_peak, "unit": "GB/s", "frac": 8.0 * n * n / t_solve / 1e9 / hbm_peak,
                           "note": "algorithmic bytes 8 N^2: two sweeps over the 4 N^2-byte triangle"},
        "predict_mean_kernel_evals_per_s": len(Xs_local) * n / t_mean_full,
        "predict_mean_note": "predict() uses tgp_predict_mean_trunc (Hilbert-sorted blocks, pairs with correlation "
                             "< 1e-40 skipped); kernel_evals_per_s is the untruncated kernel evaluating all M x N pairs",
    }
    del ws
    torch.cuda.empty_cache()
    return short, long


def desc_theta(treegp, desc, template):
    """theta of the fitted kernel from its descriptor (for the record only)."""
    inv = np.array([[desc.m00, desc.m01], [desc.m01, desc.m11]])
    k = treegp.eval_kernel("%r * AnisotropicVonKarman(invLam=array([[%.17g, %.17g], [%.17g, %.17g]]))" % (
        desc.amp, inv[0, 0], inv[0, 1], inv[1, 0], inv[1, 1]))
    return k.theta


def run_cfg2(args, treegp, backend, ctx):
    """configs[1]: 2-D AnisotropicRBF GP, N = 10,000, optimizer='log-likelihood' (FP64 Cholesky + marginal
    likelihood inside scipy's L-BFGS-B loop).  With more than one rank the (n_theta + 1) probes of every
    forward-difference gradient are dealt to the ranks (replicated data, one tiny all-reduce per gradient:
    treegp_b200/log_likelihood.py, SURVEY 8e) and every rank must arrive at the identical theta-hat."""
    import torch
    from treegp_b200.two_pcf import get_correlation_length_matrix

    rank, world, dev, barrier, max_over_ranks, tdist = (ctx[k] for k in ("rank", "world", "dev", "barrier",
                                                                          "max_over_ranks", "tdist"))
    rng = np.random.default_rng(7)
    n = 10_000
    L = 80.0 * np.sqrt(n / 16000.0)
    inv = np.linalg.inv(get_correlation_length_matrix(0.5, 0.2, 0.2))
    kstr = "4.0 * AnisotropicRBF(invLam=array([[%.17g, %.17g], [%.17g, %.17g]]))" % (inv[0, 0], inv[0, 1], inv[1, 0], inv[1, 1])
    X = rng.uniform(-L / 2, L / 2, size=(n, 2))
    kern = treegp.eval_kernel(kstr)
    y, y_err = treegp.sample_grf(kern, X, noise=0.01, seed=8)
    llmod = sys.modules["treegp_b200.log_likelihood"]
    out = {}

    def fit(distributed):
        llmod.DISTRIBUTED_FD = distributed
        gp = treegp.GPInterpolation(kernel=kstr, optimizer="log-likelihood", normalize=True)
        gp.initialize(X, y, y_err=y_err)
        barrier()
        t0 = time.perf_counter()
        gp.solve()
        torch.cuda.synchronize()
        dt = max_over_ranks(time.perf_counter() - t0)
        llmod.DISTRIBUTED_FD = False
        return gp, dt

    fit(False) if world == 1 else None
    gp, t_fit = fit(world > 1)
    nev = gp._optimizer.n_evaluations
    out["cfg2_fit_s"] = t_fit
    out["cfg2_evals_this_rank"] = nev
    out["cfg2_s_per_eval"] = t_fit / max(nev, 1) if world == 1 else None
    out["cfg2_logL"] = float(gp._optimizer._logL)
    out["cfg2_theta"] = [float(v) for v in gp.kernel.theta]
    if world > 1:
        th = torch.tensor(gp.kernel.theta, dtype=torch.float64, device=dev)
        every = [torch.zeros_like(th) for _ in range(world)]
        tdist.all_gather(every, th)
        out["cfg2_theta_identical_on_all_ranks"] = bool(all(torch.equal(every[0], e) for e in every))
        out["cfg2_fd_probes"] = "dealt over %d ranks" % world
    return out


def rff_field(X, inv, sigma, features=384, seed=3):
    """Random-Fourier-feature synthesis of a zero-mean Gaussian field with kernel sigma^2 exp(-d^T inv d / 2)."""
    rng = np.random.default_rng(seed)
    Lc = np.linalg.cholesky(inv)
    omega = rng.normal(size=(features, 2)) @ Lc.T
    phase = rng.uniform(0, 2 * np.pi, size=features)
    y = np.zeros(len(X))
    for a in range(0, features, 64):
        y += np.cos(X @ omega[a:a + 64].T + phase[a:a + 64]).sum(axis=1)
    return sigma * np.sqrt(2.0 / features) * y


def run_cfg5(args, treegp, backend, ctx):
    """configs[4]: N = 200,000, robust 2PCF hyper-parameter fit with 100 batched bootstrap resamples plus the meanify
    mean function: meanify (host, O(N)) -> FITS table -> GPInterpolation.initialize (KNN(4) mean subtraction on the
    device) -> comp_2pcf + comp_xi_covariance(100) + robust_2dfit; then the public solve() with the reference's own
    resample count (444 for nbins = 21)."""
    import torch
    from treegp_b200.two_pcf import get_correlation_length_matrix, robust_2dfit

    out = {}
    n = 200_000
    Lf = 1000.0 * np.sqrt(n / 1e6)
    rng = np.random.default_rng(11)
    X = rng.uniform(-Lf / 2, Lf / 2, size=(n, 2))
    size, g1, g2, sigma, noise = 8.0, 0.2, 0.1, 1.0, 0.05
    inv = np.linalg.inv(get_correlation_length_matrix(size, g1, g2))
    mean_of = lambda P_: 0.5 * np.sin(P_[:, 0] / 70.0) * np.cos(P_[:, 1] / 90.0)
    y = rff_field(X, inv, sigma) + mean_of(X) + rng.normal(scale=noise, size=n)
    y_err = np.full(n, noise)
    # the mean function is what survives the average over many exposures: five more realisations of the random
    # field (other positions, other phases) enter the meanify grid next to the field that is fitted
    others = []
    for s_ in range(5):
        Xo = rng.uniform(-Lf / 2, Lf / 2, size=(n, 2))
        others.append((Xo, rff_field(Xo, inv, sigma, seed=100 + s_) + mean_of(Xo) + rng.normal(scale=noise, size=n)))
    kstr = "1.0 * AnisotropicRBF(invLam=array([[%.17g, %.17g], [%.17g, %.17g]]))" % (inv[0, 0], inv[0, 1], inv[1, 0], inv[1, 1])
    tmp = os.path.join(tempfile.mkdtemp(prefix="tgp_bench_"), "mean_gp.fits")
    max_sep, B = 30.0, 100

    def run():
        t = {}
        t0 = time.perf_counter()
        mf = treegp.meanify(bin_spacing=Lf / 50.0, statistics="mean")
        mf.add_field(X, y)
        for Xo, yo in others:
            mf.add_field(Xo, yo)
        mf.meanify()
        mf.save_results(name_output=tmp)
        t["meanify_s"] = time.perf_counter() - t0
        t1 = time.perf_counter()
        gp = treegp.GPInterpolation(kernel=kstr, optimizer="anisotropic", normalize=True, average_fits=tmp, n_neighbors=4,
                                    nbins=21, min_sep=0.0, max_sep=max_sep, p0=[6.0, 0.0, 0.0])
        gp.initialize(X, y, y_err=y_err)          # KNN(4) lookup of the mean grid for all N points
        torch.cuda.synchronize()
        t["initialize_knn_mean_s"] = time.perf_counter() - t1
        resid = gp._y - gp._mean - gp._spatial_average
        t2 = time.perf_counter()
        tp = treegp.two_pcf(X, resid, y_err, 0.0, max_sep, nbins=21, anisotropic=True, robust_fit=True, p0=[6.0, 0.0, 0.0])
        xi, dist_, coord, mask = tp.comp_2pcf(X, resid, y_err)
        torch.cuda.synchronize()
        t["pair_count_s"] = time.perf_counter() - t2
        t3 = time.perf_counter()
        cov = tp.comp_xi_covariance(n_bootstrap=B, mask=mask, seed=610639139)
        torch.cuda.synchronize()
        t["bootstrap_%d_s" % B] = time.perf_counter() - t3
        t4 = time.perf_counter()
        # 100 resamples of 221 pixels give a singular covariance: the robust fit of this config uses its diagonal
        W = np.diag(1.0 / np.diag(cov))
        rob = robust_2dfit(gp.kernel_template, xi, coord[:, 0], coord[:, 1], W, mask=mask)
        rob.minimize_minuit(p0=[6.0, 0.0, 0.0])
        t["robust_fit_s"] = time.perf_counter() - t4
        t["total_s"] = time.perf_counter() - t0
        return t, rob.result, gp

    run()
    t, result, gp = run()
    out["cfg5_total_s"] = t["total_s"]
    out["cfg5_breakdown_s"] = t
    out["cfg5_fit_sigma_size_g1_g2_offset"] = [float(v) for v in result]
    out["cfg5_truth_sigma_size_g1_g2"] = [sigma, size, g1, g2]
    pairs = n * (n - 1) / 2
    out["cfg5_bootstrap_resample_pairs_per_s"] = B * pairs / t["bootstrap_%d_s" % B]
    # the round-1 bootstrap record, for comparison: iid field, default max_sep (half the diagonal), 100 resamples
    tq = treegp.two_pcf(X, rng.normal(size=n), np.zeros(n), 0.0, np.sqrt(2.0) * Lf / 2.0, nbins=21, anisotropic=True)
    tq.comp_xi_covariance(n_bootstrap=2, mask=None, seed=1)
    torch.cuda.synchronize()
    backend.bootbin_stats(reset=True)
    t0 = time.perf_counter()
    tq.comp_xi_covariance(n_bootstrap=B, mask=None, seed=610639139)
    torch.cuda.synchronize()
    out["cfg5_bootstrap100_default_maxsep_s"] = time.perf_counter() - t0
    out["cfg5_bootstrap_paths_blocks"] = backend.bootbin_stats()
    # the same resamples as independent weighted catalogues of one tgp_pairbin launch (the round-1 batch)
    tq.SHARED_BOOTSTRAP = False
    tq.comp_xi_covariance(n_bootstrap=2, mask=None, seed=1)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    tq.comp_xi_covariance(n_bootstrap=B, mask=None, seed=610639139)
    torch.cuda.synchronize()
    out["cfg5_bootstrap100_default_maxsep_per_catalogue_s"] = time.perf_counter() - t0
    tq.SHARED_BOOTSTRAP = True
    # the public path: solve() = pair count + 444 resamples (fsolve, two_pcf.py:375-383) + robust fit
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    gp.solve()
    torch.cuda.synchronize()
    out["cfg5_solve_444_resamples_s"] = time.perf_counter() - t0
    out["cfg5_solve_result"] = [float(v) for v in gp._optimizer._results_robust]
    return out


def run_bootstrap_sharded(args, treegp, backend, dist, ctx):
    """N > 1: the 100-resample bootstrap of configs[4] (iid field, N = 200k, default max_sep) with the work items of
    tgp_bootbin_twod dealt to the ranks and ONE all-reduce of the per-resample sums (torch.distributed / NCCL)."""
    import torch

    rank, world, dev, barrier, max_over_ranks = (ctx[k] for k in ("rank", "world", "dev", "barrier", "max_over_ranks"))
    n, B = 200_000, 100
    Lf = 1000.0 * np.sqrt(n / 1e6)
    rng = np.random.default_rng(11)
    X = rng.uniform(-Lf / 2, Lf / 2, size=(n, 2))
    tq = treegp.two_pcf(X, rng.normal(size=n), np.zeros(n), 0.0, np.sqrt(2.0) * Lf / 2.0, nbins=21, anisotropic=True)
    tq.group = dist.WORLD
    tq.comp_xi_covariance(n_bootstrap=2, mask=None, seed=1)
    torch.cuda.synchronize()
    barrier()
    t0 = time.perf_counter()
    cov = tq.comp_xi_covariance(n_bootstrap=B, mask=None, seed=610639139)
    torch.cuda.synchronize()
    dt = max_over_ranks(time.perf_counter() - t0)
    return {"cfg5_bootstrap100_default_maxsep_s": dt, "cfg5_bootstrap_cov_trace": float(np.trace(cov)),
            "cfg5_bootstrap_sharding": "work items of tgp_bootbin_twod over %d ranks + one all-reduce of the sums" % world}


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
