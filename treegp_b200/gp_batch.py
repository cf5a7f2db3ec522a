"""GPInterpolationBatch: many independent small Gaussian-process problems (e.g. one PSF parameter of one exposure
each) fitted, solved and predicted together on the B200.

A problem of a few hundred to a few thousand points leaves the GPU idle: its factorisation is a chain of small
launches.  Here every launch carries all problems (tgp_loglike_batch / tgp_predict_mean_batch), and the
"log-likelihood" fit runs the B scipy L-BFGS-B searches in lock step, so that each round of likelihood evaluations of
all live problems is one batched device call.  Per problem the class behaves like ``GPInterpolation`` with the same
arguments: a problem's likelihood values are those of the single (dense) path bit for bit, so the lock-step fit
reproduces each problem's own fit exactly.
"""
import copy
import queue
import threading

import numpy as np
import torch
from scipy import optimize

from . import _cabi, backend
from .kernels import descriptor_params, eval_kernel, lower, lower_jacobian
from .log_likelihood import log_likelihood
from .two_pcf import two_pcf

OPTIMIZERS = ["anisotropic", "two-pcf", "log-likelihood", "none"]
_ABORT = object()


def lockstep_minimize(evaluate, x0s, jac=False):
    """Run one ``scipy.optimize.minimize(f_b, x0s[b], method="L-BFGS-B")`` per problem, exactly as
    ``log_likelihood.optimizer`` does (no bounds, scipy's forward-difference gradient), with the objective values of
    all problems computed together.  With jac=True each search is ``minimize(f_b, x0s[b], method="L-BFGS-B",
    jac=True)`` and ``evaluate`` returns one (value, gradient) pair per request, as with ANALYTIC_GRADIENT.

    Each search runs in a worker thread whose objective only posts its theta and waits.  The calling thread collects
    one request from every live search, calls ``evaluate(indices, thetas)`` (a sequence of objective values, one per
    request) and replies; searches that have finished drop out.  Workers never touch the device.  All threads are
    joined before this returns, also when ``evaluate`` or a search raises (the first error is re-raised).  Returns the
    list of minimisers."""
    B = len(x0s)
    requests = queue.Queue()
    replies = [queue.Queue() for _ in range(B)]
    results = [None] * B

    def worker(b):
        def fun(theta):
            requests.put(("eval", b, np.array(theta, dtype=float)))
            v = replies[b].get()
            if v is _ABORT:
                raise RuntimeError("lock-step search aborted")
            return v

        try:
            requests.put(("done", b, optimize.minimize(fun, x0s[b], method="L-BFGS-B", jac=jac)["x"]))
        except BaseException as e:  # noqa: BLE001  (handed to the calling thread, which re-raises)
            requests.put(("error", b, e))

    threads = [threading.Thread(target=worker, args=(b,), daemon=True) for b in range(B)]
    for t in threads:
        t.start()
    live, pending, error = B, [], None
    try:
        while live:
            msgs = [requests.get() for _ in range(live)]   # every live search posts exactly one message per round
            pending = [(b, th) for kind, b, th in msgs if kind == "eval"]
            for kind, b, payload in msgs:
                if kind == "done":
                    results[b] = payload
                elif kind == "error" and error is None:
                    error = payload
            live = len(pending)
            if error is not None:
                break
            if pending:
                values = list(evaluate([b for b, _ in pending], [th for _, th in pending]))
                if len(values) != len(pending):
                    raise ValueError("evaluate returned %d values for %d requests" % (len(values), len(pending)))
                for (b, _), v in zip(pending, values):
                    replies[b].put((float(v[0]), np.array(v[1], dtype=float)) if jac else float(v))
                pending = []
    except BaseException as e:  # noqa: BLE001
        error = e
    finally:
        if error is not None:
            for b, _ in pending:   # release the searches still waiting for a value; each then posts its error
                replies[b].put(_ABORT)
            for _ in pending:
                requests.get()
        for t in threads:
            t.join()
    if error is not None:
        raise error
    return results


class GPInterpolationBatch(object):
    """B independent Gaussian-process interpolations of scalar surfaces, put through the device together.

    Constructor keywords mean what they mean in ``GPInterpolation``:

    kernel          one kernel string shared by all problems (each gets its own copy), or a list of B strings
    optimizer       "none", "two-pcf", "anisotropic" (the per-problem 2-point-function fits, run one after the other)
                    or "log-likelihood" (the B likelihood searches in lock step, one batched evaluation per round)
    normalize, p0, white_noise, nbins, min_sep, max_sep  as in GPInterpolation

    Every problem has at most TGP_BATCH_MAX_N = 4096 points (use GPInterpolation above that) and one ndim applies to
    all.  The factorisation is always dense.  The fitted kernels are in ``kernels``."""

    WORK_BUDGET = 4 << 30   # bytes of device workspace per batched call; larger batches run in several chunks

    def __init__(self, kernel="RBF(1)", optimizer="two-pcf", normalize=True, p0=[3000.0, 0.0, 0.0], white_noise=0.0,
                 nbins=20, min_sep=None, max_sep=None):
        if optimizer not in OPTIMIZERS:
            raise ValueError("Only anisotropic, two-pcf, log-likelihood and none are supported for optimizer. "
                             "Current value: %s" % (optimizer,))
        if isinstance(kernel, str):
            self.kernel_template = eval_kernel(kernel)
        elif isinstance(kernel, (list, tuple)) and len(kernel) > 0 and all(isinstance(k, str) for k in kernel):
            self.kernel_template = [eval_kernel(k) for k in kernel]
        else:
            raise TypeError("kernel should be a string or a list of B strings")
        self.optimizer = optimizer
        self.normalize = normalize
        self.p0_robust_fit = p0
        self.white_noise = white_noise
        self.nbins = nbins
        self.min_sep = min_sep
        self.max_sep = max_sep
        self._solved = None

    def initialize(self, Xs, ys, y_errs=None):
        """Attach B problems: lists of positions (N_b, ndim), values (N_b,) and optional errors (N_b,).  Per problem
        what GPInterpolation.initialize does: a fresh copy of the kernel, zero errors when none are given, the white
        noise added in quadrature and the normalising mean."""
        B = len(Xs)
        if B == 0 or len(ys) != B or (y_errs is not None and len(y_errs) != B):
            raise ValueError("Xs, ys and y_errs must be lists of the same, non-zero length (%d, %d, %s)"
                             % (B, len(ys), "None" if y_errs is None else len(y_errs)))
        templates = self.kernel_template if isinstance(self.kernel_template, list) else [self.kernel_template] * B
        if len(templates) != B:
            raise ValueError("%d kernel strings for %d problems" % (len(templates), B))
        ndims = set()
        for b in range(B):
            X, y = np.asarray(Xs[b]), np.asarray(ys[b])
            if y.ndim != 1:
                raise ValueError("problem %d: y must be 1-D (one output per problem); got shape %r" % (b, y.shape))
            if X.ndim != 2 or X.shape[0] != len(y) or len(y) == 0:
                raise ValueError("problem %d: X must have shape (N, ndim) with N = len(y) >= 1; got %r" % (b, X.shape))
            if y_errs is not None and y_errs[b] is not None and np.shape(y_errs[b]) != y.shape:
                raise ValueError("problem %d: y_err must have the shape of y" % b)
            if len(y) > _cabi.BATCH_MAX_N:
                raise ValueError("problem %d has %d points; a batch takes at most %d per problem (TGP_BATCH_MAX_N) -- "
                                 "use GPInterpolation for it" % (b, len(y), _cabi.BATCH_MAX_N))
            ndims.add(X.shape[1])
        if len(ndims) != 1:
            raise ValueError("every problem of a batch must have the same ndim; got %s" % sorted(ndims))
        self.kernels = [copy.deepcopy(t) for t in templates]
        self._X, self._y, self._y_err, self._mean, self._spatial_average = [], [], [], [], []
        for b in range(B):
            y = ys[b]
            y_err = np.zeros_like(y) if y_errs is None or y_errs[b] is None else y_errs[b]
            self._X.append(Xs[b])
            self._y.append(y)
            self._spatial_average.append(np.zeros(len(Xs[b][:, 0])))
            if self.white_noise > 0:
                y_err = np.sqrt(np.array(y_err, dtype=float) ** 2 + self.white_noise ** 2)
            self._y_err.append(y_err)
            self._mean.append(np.mean(y - self._spatial_average[b]) if self.normalize else 0.0)
        self._dev = None
        self._solved = None

    def _residual(self, b):
        return self._y[b] - self._mean[b] - self._spatial_average[b]

    def _device_data(self):
        """Concatenated X, residual y and y_err^2 of all problems on the device (built once per initialize)."""
        if self._dev is None:
            X = torch.cat([backend.as_points(X) for X in self._X])
            y = backend.to_device(np.concatenate([np.asarray(self._residual(b), dtype=np.float64).reshape(-1)
                                                  for b in range(len(self._X))]))
            e2 = backend.to_device(np.concatenate([np.asarray(e, dtype=np.float64).reshape(-1) ** 2
                                                   for e in self._y_err]))
            sizes = [len(y) for y in self._y]
            self._dev = (X, y, e2, sizes, backend.batch_offsets(sizes))
        return self._dev

    def _batched(self, indices, descs, call, name):
        """One batched device call `call` (backend.loglike_batch or loglike_grad_batch, chunked by WORK_BUDGET) over
        the problems `indices` whose descriptor in `descs` is finite; the others launch nothing (as
        log_likelihood.log_likelihood).  Returns (the positions in `indices` that ran, their out rows on the host)."""
        X, y, e2, sizes, off = self._device_data()
        run = [i for i, d in enumerate(descs) if np.all(np.isfinite(descriptor_params(d)))]
        if not run:
            return run, None
        probs = [indices[i] for i in run]
        if probs == list(range(len(sizes))):
            Xr, yr, er = X, y, e2
        else:
            rows = torch.as_tensor(np.concatenate([np.arange(off[b], off[b + 1]) for b in probs]), device=X.device)
            Xr, yr, er = X[rows].contiguous(), y[rows].contiguous(), e2[rows].contiguous()
        out, info, _ = call(Xr, yr, er, [sizes[b] for b in probs], [descs[i] for i in run],
                            budget_bytes=self.WORK_BUDGET)
        out = out.cpu().numpy()
        if np.any(out[:, 0] != out[:, 0]):   # NaN marks info < 0: an internal synchronisation timeout, never a -inf
            raise _cabi.TgpError("%s: internal synchronisation timed out (info = %r)"
                                 % (name, info.cpu().numpy().tolist()))
        return run, out

    def _loglike(self, indices, kernels):
        """logL of the problems `indices` for `kernels`: one batched call for those whose descriptor is finite, -inf
        without a launch for the others."""
        ndim = self._device_data()[0].shape[1]
        values = np.full(len(indices), -np.inf)
        run, out = self._batched(indices, [lower(k, ndim) for k in kernels], backend.loglike_batch,
                                 "tgp_loglike_batch")
        if run:
            values[run] = out[:, 0]
        return values

    def _loglike_and_gradient(self, indices, kernels):
        """(logL, d logL / d theta) of the problems `indices` for `kernels`: one batched value-and-gradient call
        (tgp_loglike_grad_batch) for those whose descriptor is finite; -inf and a zero gradient without a launch for
        the others, and -inf with a zero gradient where K is not positive definite (as
        log_likelihood.log_likelihood_and_gradient).  A list of (value, gradient) pairs."""
        ndim = self._device_data()[0].shape[1]
        descs, jacs = zip(*[lower_jacobian(k, ndim) for k in kernels])
        results = [(-np.inf, np.zeros(J.shape[1])) for J in jacs]
        run, out = self._batched(indices, descs, backend.loglike_grad_batch, "tgp_loglike_grad_batch")
        for i, o in zip(run, out if run else []):
            results[i] = (float(o[0]), jacs[i].T @ o[3:3 + jacs[i].shape[0]])   # the gradient is 0 where logL = -inf
        return results

    def solve(self):
        """Fit every problem's kernel with the configured optimizer.  With log_likelihood.ANALYTIC_GRADIENT set (the
        switch GPInterpolation honours), the "log-likelihood" searches use the analytic gradient: one batched
        value-and-gradient call per round."""
        B = len(self._X)
        self._init_theta = [copy.deepcopy(k).theta for k in self.kernels]
        self._solved = None
        if self.optimizer == "log-likelihood" and log_likelihood.ANALYTIC_GRADIENT:
            def evaluate_jac(indices, thetas):
                vg = self._loglike_and_gradient(indices, [self.kernels[b].clone_with_theta(t)
                                                          for b, t in zip(indices, thetas)])
                return [(-v, -g) for v, g in vg]

            best = lockstep_minimize(evaluate_jac, [k.theta for k in self.kernels], jac=True)
            self.kernels = [self.kernels[b].clone_with_theta(best[b]) for b in range(B)]
        elif self.optimizer == "log-likelihood":
            def evaluate(indices, thetas):
                return -self._loglike(indices, [self.kernels[b].clone_with_theta(t) for b, t in zip(indices, thetas)])

            best = lockstep_minimize(evaluate, [k.theta for k in self.kernels])
            self.kernels = [self.kernels[b].clone_with_theta(best[b]) for b in range(B)]
        elif self.optimizer in ["two-pcf", "anisotropic"]:
            for b in range(B):
                fit = two_pcf(self._X[b], self._residual(b), self._y_err[b], self.min_sep, self.max_sep,
                              nbins=self.nbins, anisotropic=self.optimizer == "anisotropic",
                              robust_fit=self.optimizer == "anisotropic", p0=self.p0_robust_fit)
                self.kernels[b] = fit.optimizer(self.kernels[b])

    def _ensure_solved(self):
        """alpha = K^-1 y of every problem for the current kernels (one batched call), cached until the next fit."""
        if self._solved is not None:
            return self._solved
        X, y, e2, sizes, _ = self._device_data()
        descs = [lower(k, X.shape[1]) for k in self.kernels]
        for b, d in enumerate(descs):
            if not np.all(np.isfinite(descriptor_params(d))):
                raise np.linalg.LinAlgError("problem %d: the kernel has non-finite parameters" % b)
        _, info, alpha = backend.loglike_batch(X, y, e2, sizes, descs, want_alpha=True, budget_bytes=self.WORK_BUDGET)
        info = info.cpu().numpy()
        if np.any(info < 0):
            raise _cabi.TgpError("tgp_loglike_batch: internal synchronisation timed out (info = %r)" % info.tolist())
        bad = np.flatnonzero(info > 0)
        if len(bad):
            raise np.linalg.LinAlgError("problem %d: %d-th leading minor of the array is not positive definite"
                                        % (bad[0], info[bad[0]]))
        self._solved = (descs, alpha)
        return self._solved

    def predict(self, Xs_new, return_cov=False):
        """Posterior means at the positions Xs_new[b] (M_b, ndim) of every problem: a list of B arrays."""
        if return_cov:
            raise ValueError("GPInterpolationBatch predicts means only; use GPInterpolation for a covariance")
        if len(Xs_new) != len(self._X):
            raise ValueError("need one set of positions per problem (%d for %d problems)" % (len(Xs_new), len(self._X)))
        descs, alpha = self._ensure_solved()
        X, _, _, sizes, _ = self._device_data()
        ssizes = [len(np.asarray(x)) for x in Xs_new]
        Xs = torch.cat([backend.as_points(x) for x in Xs_new])
        mean = backend.predict_mean_batch(Xs, ssizes, X, sizes, descs, alpha).cpu().numpy()
        soff = backend.batch_offsets(ssizes)
        return [mean[soff[b]:soff[b + 1]] + self._mean[b] + np.zeros(ssizes[b]) for b in range(len(sizes))]

    def return_log_likelihood(self, thetas=None):
        """Marginal log-likelihood of every problem for its current kernel, or for thetas[b] if given: an array of B
        values from one batched call."""
        kernels = [copy.deepcopy(k) for k in self.kernels]
        if thetas is not None:
            kernels = [k.clone_with_theta(t) for k, t in zip(kernels, thetas)]
        return self._loglike(list(range(len(kernels))), kernels)
