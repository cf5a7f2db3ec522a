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
from .gp_interp import TWO_PCF_NEEDS_1D_Y
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
    """B independent Gaussian-process interpolations, put through the device together.  Each problem has one scalar
    field, or r fields (1 <= r <= TGP_MAX_RHS, the same r for all problems) that share its kernel, as a 2-D y does
    in ``GPInterpolation``.

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
        """Attach B problems: lists of positions (N_b, ndim), values (N_b,) -- or (N_b, r) for r outputs sharing the
        problem's kernel, one r for every problem -- and optional errors (N_b,), shared by the outputs.  Per problem
        what GPInterpolation.initialize does: a fresh copy of the kernel, zero errors when none are given, the white
        noise added in quadrature and the normalising mean (one per output)."""
        B = len(Xs)
        if B == 0 or len(ys) != B or (y_errs is not None and len(y_errs) != B):
            raise ValueError("Xs, ys and y_errs must be lists of the same, non-zero length (%d, %d, %s)"
                             % (B, len(ys), "None" if y_errs is None else len(y_errs)))
        templates = self.kernel_template if isinstance(self.kernel_template, list) else [self.kernel_template] * B
        if len(templates) != B:
            raise ValueError("%d kernel strings for %d problems" % (len(templates), B))
        ndims = set()
        shape0 = np.shape(ys[0])
        for b in range(B):
            X, y = np.asarray(Xs[b]), np.asarray(ys[b])
            if y.ndim not in (1, 2) or y.ndim != len(shape0):
                raise ValueError("problem %d: y has shape %r; a batch takes 1-D ys (N_b,) or 2-D ys (N_b, r), the same "
                                 "for all problems (problem 0: %r)" % (b, y.shape, shape0))
            if y.ndim == 2 and not (1 <= y.shape[1] <= _cabi.MAX_RHS and y.shape[1] == shape0[1]):
                raise ValueError("problem %d: y has %d outputs; a batch takes one r, 1 <= r <= %d (TGP_MAX_RHS), for "
                                 "all problems (problem 0: %d)" % (b, y.shape[1], _cabi.MAX_RHS, shape0[1]))
            if X.ndim != 2 or X.shape[0] != len(y) or len(y) == 0:
                raise ValueError("problem %d: X must have shape (N, ndim) with N = len(y) >= 1; got %r" % (b, X.shape))
            if y_errs is not None and y_errs[b] is not None and np.shape(y_errs[b]) != (len(y),):
                raise ValueError("problem %d: y_err must have shape (N,) = (%d,), shared by the outputs; got %r"
                                 % (b, len(y), np.shape(y_errs[b])))
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
            multi = np.ndim(y) == 2
            y_err = (np.zeros(len(y)) if multi else np.zeros_like(y)) if y_errs is None or y_errs[b] is None else y_errs[b]
            self._X.append(Xs[b])
            self._y.append(y)
            self._spatial_average.append(np.zeros(np.shape(y)))
            if self.white_noise > 0:
                y_err = np.sqrt(np.array(y_err, dtype=float) ** 2 + self.white_noise ** 2)
            self._y_err.append(y_err)
            if not self.normalize:
                self._mean.append(0.0)
            elif multi:   # column by column, as GPInterpolation.initialize: each output's mean as on its own
                res = np.asarray(y - self._spatial_average[b])
                self._mean.append(np.array([np.mean(np.ascontiguousarray(res[:, c])) for c in range(res.shape[1])]))
            else:
                self._mean.append(np.mean(y - self._spatial_average[b]))
        self._dev = None
        self._solved = None

    def _residual(self, b):
        return self._y[b] - self._mean[b] - self._spatial_average[b]

    def _device_data(self):
        """Concatenated X, residual y and y_err^2 of all problems on the device (built once per initialize)."""
        if self._dev is None:
            X = torch.cat([backend.as_points(X) for X in self._X])
            y = backend.to_device(np.concatenate([np.asarray(self._residual(b), dtype=np.float64)
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
        if np.ndim(self._y[0]) == 2 and self.optimizer in ["two-pcf", "anisotropic"]:
            raise ValueError(TWO_PCF_NEEDS_1D_Y)
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

    def _descriptors(self):
        """Every problem's kernel descriptor; LinAlgError naming the first problem whose kernel is not finite."""
        ndim = self._X[0].shape[1]
        descs = [lower(k, ndim) for k in self.kernels]
        for b, d in enumerate(descs):
            if not np.all(np.isfinite(descriptor_params(d))):
                raise np.linalg.LinAlgError("problem %d: the kernel has non-finite parameters" % b)
        return descs

    @staticmethod
    def _raise_on_info(info, name):
        """TgpError for info < 0, LinAlgError naming the first problem whose K is not positive definite."""
        info = info.cpu().numpy()
        if np.any(info < 0):
            raise _cabi.TgpError("%s: internal synchronisation timed out (info = %r)" % (name, info.tolist()))
        bad = np.flatnonzero(info > 0)
        if len(bad):
            raise np.linalg.LinAlgError("problem %d: %d-th leading minor of the array is not positive definite"
                                        % (bad[0], info[bad[0]]))

    def _ensure_solved(self):
        """alpha = K^-1 y of every problem for the current kernels (one batched call), cached until the next fit."""
        if self._solved is not None:
            return self._solved
        descs = self._descriptors()
        X, y, e2, sizes, _ = self._device_data()
        _, info, alpha = backend.loglike_batch(X, y, e2, sizes, descs, want_alpha=True, budget_bytes=self.WORK_BUDGET)
        self._raise_on_info(info, "tgp_loglike_batch")
        self._solved = (descs, alpha)
        return self._solved

    def _check_positions(self, Xs_new):
        """ValueError, before any device work, unless Xs_new holds one (M_b, ndim) array per problem."""
        if len(Xs_new) != len(self._X):
            raise ValueError("need one set of positions per problem (%d for %d problems)" % (len(Xs_new), len(self._X)))
        ndim = self._X[0].shape[1]
        for b, x in enumerate(Xs_new):
            if np.ndim(x) != 2 or np.shape(x)[1] != ndim:
                raise ValueError("problem %d: positions must have shape (M, %d); got %r" % (b, ndim, np.shape(x)))

    def predict(self, Xs_new, return_cov=False):
        """Posterior means at the positions Xs_new[b] (M_b, ndim) of every problem: a list of B arrays, (M_b,), or
        (M_b, r) for r outputs."""
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
        return [mean[soff[b]:soff[b + 1]] + self._mean[b] + np.zeros((ssizes[b],) + mean.shape[1:])
                for b in range(len(sizes))]

    def predict_var(self, Xs_new):
        """Posterior means and DIAGONAL predictive variances at the positions Xs_new[b] (M_b, ndim) of every problem:
        (means, vars), two lists of B arrays.  The means are predict's; the variances are what
        GPInterpolation.predict_var returns for the problem, bit for bit with its dense solve (residual space: the
        normalising mean does not enter).  All problems' test points go through one batched call
        (tgp_predict_var_batch), which factorises into a workspace of its own.  With r outputs the means are (M_b, r)
        and the variances (M_b,), shared by the outputs: they do not depend on y, so one output is factorised."""
        self._check_positions(Xs_new)
        means = self.predict(Xs_new)
        descs, _ = self._ensure_solved()
        X, y, e2, sizes, _ = self._device_data()
        ssizes = [len(m) for m in means]
        Xs = torch.cat([backend.as_points(x) for x in Xs_new])
        y1 = y if y.dim() == 1 else y[:, 0].contiguous()
        var, info = backend.predict_var_batch(Xs, ssizes, X, y1, e2, sizes, descs, budget_bytes=self.WORK_BUDGET)
        self._raise_on_info(info, "tgp_loglike_batch")
        var = var.cpu().numpy()
        soff = backend.batch_offsets(ssizes)
        return means, [var[soff[b]:soff[b + 1]] for b in range(len(sizes))]

    def loo_predict(self):
        """Leave-one-out predictions at every training point of every problem, without refitting: (means, vars), two
        lists of B arrays in each problem's own order, as GPInterpolation.loo_predict gives them -- mean_i = y_i -
        alpha_i / Z_ii plus the normalising mean, var_i = 1 / Z_ii - y_err_i^2, Z = (K + diag(y_err^2))^-1.  One
        batched call (tgp_loo_batch) factorises and inverts every problem in a workspace of its own.  With r outputs
        the means are (N_b, r), mean_ic = y_ic - alpha_ic / Z_ii, and the variances (N_b,)."""
        descs = self._descriptors()
        X, y, e2, sizes, off = self._device_data()
        mean, var, info = backend.loo_batch(X, y, e2, sizes, descs, budget_bytes=self.WORK_BUDGET)
        self._raise_on_info(info, "tgp_loo_batch")
        mean, var = mean.cpu().numpy(), var.cpu().numpy()
        return ([mean[off[b]:off[b + 1]] + self._mean[b] + self._spatial_average[b] for b in range(len(sizes))],
                [var[off[b]:off[b + 1]] for b in range(len(sizes))])

    def return_log_likelihood(self, thetas=None):
        """Marginal log-likelihood of every problem for its current kernel, or for thetas[b] if given: an array of B
        values from one batched call (with r outputs the joint value, the sum over the outputs)."""
        kernels = [copy.deepcopy(k) for k in self.kernels]
        if thetas is not None:
            kernels = [k.clone_with_theta(t) for k, t in zip(kernels, thetas)]
        return self._loglike(list(range(len(kernels))), kernels)
