"""Marginal log-likelihood of a Gaussian process and its maximisation, evaluated on the B200.

Host-side mirror of /root/reference/treegp/log_likelihood.py (class ``log_likelihood``: same
constructor, ``log_likelihood(kernel)``, ``optimizer(kernel)``, attributes ``_kernel`` and ``_logL``).
The body of one evaluation (log_likelihood.py:29-37: K build, Cholesky, solve, chi2, log-det) is a
single C-ABI call, ``tgp_loglike``; X, y, y_err^2 and the N x N workspace stay resident on the
device for the whole L-BFGS-B search (40-120 evaluations per fit, SURVEY.md section 3.2).
"""
import copy

import numpy as np
from scipy import optimize

from . import backend
from .kernels import descriptor_params, lower, lower_jacobian

# Multi-GPU (SURVEY.md section 8e): the (n_theta + 1) likelihood evaluations of one forward-difference gradient
# are independent.  With DISTRIBUTED_FD = True (or env TREEGP_B200_DIST_FD=1) and an initialised process group,
# every rank runs the same L-BFGS-B loop on replicated data and evaluates only its share of the probes; the
# values are exchanged with one tiny all-reduce per gradient, so all ranks take identical steps.  Opt-in
# because every rank of the group must then call optimizer() together.
DISTRIBUTED_FD = False
_FD_STEP = 1e-8  # scipy's default absolute forward-difference step for L-BFGS-B


class log_likelihood(object):
    """Marginal log-likelihood of a GP for a kernel, and its maximiser over the kernel's theta.

    X: (n, 1|2) positions; y: (n,) residual field values; y_err: (n,) one-sigma errors added in quadrature
    on the diagonal.  Same constructor as the reference class of the same name.

    y of shape (n, r), 1 <= r <= 8 (extension): r outputs sharing the kernel and y_err.  The log-likelihood is then the
    joint value sum_c logL_c (scikit-learn's log_marginal_likelihood for multi-target y), from one factorisation.
    """

    def __init__(self, X, y, y_err):
        self.X = X
        self.ndata = len(self.X[:, 0])
        self.y = y
        self.y_err = y_err
        self._dev = None
        self.n_evaluations = 0

    def _device_state(self):
        if self._dev is None:
            Xd = backend.as_points(self.X)
            if np.ndim(self.y) == 2:   # several outputs: r extra rows ride through potrf
                yd = backend.to_device(np.asarray(self.y, dtype=np.float64))
                rows = yd.shape[1]
            else:
                yd = backend.to_device(np.asarray(self.y, dtype=np.float64).reshape(-1))
                rows = 1
            e2 = backend.to_device(np.asarray(self.y_err, dtype=np.float64).reshape(-1) ** 2)
            work = backend.alloc_matrix(self.ndata + rows, self.ndata, Xd.device)  # the outputs ride through potrf
            self._dev = (Xd, yd, e2, work)
            self._sorted_axes = {}   # backend.plan_envelope's cache: order / coordinates per sorting axis
            self._sorted_data = {}   # axis -> (X, y, y_err^2) in that order
        return self._dev

    # Factorise inside the envelope of K when the probed kernel's support is short against the field
    # (backend.plan_envelope: the points sorted along one axis; N bw^2 flop instead of N^3 / 3).  The value is the
    # same to rounding: entries of K below 1e-40 of the amplitude count as zero.
    BANDED = True

    def _envelope_inputs(self, desc):
        """(X, y, y_err^2, row_end) sorted for the envelope factorisation of this kernel, or None (dense)."""
        Xd, yd, e2, _ = self._dev
        env = backend.plan_envelope(Xd, desc, sorted_axes=self._sorted_axes) if self.BANDED else None
        if env is None:
            return None
        ax = env["axis"]
        if ax not in self._sorted_data:
            o = env["order"]
            self._sorted_data[ax] = (Xd[o].contiguous(), yd[o].contiguous(), e2[o].contiguous())
        return self._sorted_data[ax] + (env["row_end"],)

    def log_likelihood(self, kernel):
        """log p(y | X, kernel) = -chi2/2 - n/2 ln(2 pi) - ln|K|/2, or -inf when K + diag(y_err^2) is not
        positive definite.  `kernel` is a scikit-learn style kernel object."""
        Xd, yd, e2, work = self._device_state()
        desc = lower(kernel, Xd.shape[1])
        # a non-finite hyper-parameter cannot be factorised: the reference's try/except returns -inf
        # (log_likelihood.py:38-39); same outcome here without launching anything
        if not np.all(np.isfinite(descriptor_params(desc))):
            return -np.inf
        banded = self._envelope_inputs(desc)
        loglike = backend.loglike_multi if yd.dim() == 2 else backend.loglike
        if banded is None:
            out, info, _, _ = loglike(Xd, yd, e2, desc, work=work, want_alpha=False)
        else:
            out, info, _, _ = loglike(banded[0], banded[1], banded[2], desc, work=work, want_alpha=False,
                                      row_end=banded[3])
            self.n_banded_evaluations = getattr(self, "n_banded_evaluations", 0) + 1
        self.n_evaluations += 1
        value = float(out[0].item())  # -inf when the matrix is not positive definite (info > 0)
        if value != value:            # NaN marks info < 0: an internal synchronisation timeout, never a -inf
            from ._cabi import TgpError
            raise TgpError("tgp_loglike: internal synchronisation timed out (info = %d)" % int(info.item()))
        return value

    # optimizer(): L-BFGS-B with the analytic gradient of log_likelihood_and_gradient (jac=True) instead of scipy's
    # forward differences (n_theta + 1 evaluations per gradient, each component with ~1e-8 relative noise of logL)
    ANALYTIC_GRADIENT = False

    def log_likelihood_and_gradient(self, kernel):
        """(log p(y | X, kernel), d log p / d kernel.theta) from one device call (tgp_loglike_grad: the factorisation,
        the selected inverse Z = K^-1 inside its envelope and one contraction with alpha alpha^T - Z).  Same envelope
        choice and -inf rule as log_likelihood; the gradient is 0 where the value is -inf."""
        Xd, yd, e2, work = self._device_state()
        desc, J = lower_jacobian(kernel, Xd.shape[1])
        if not np.all(np.isfinite(descriptor_params(desc))):
            return -np.inf, np.zeros(J.shape[1])
        banded = self._envelope_inputs(desc)
        # several outputs: tgp_loglike_grad_multi, whose out has the sum layout (a single term's four derivatives first)
        loglike_grad = backend.loglike_grad_multi if yd.dim() == 2 else backend.loglike_grad
        if banded is None:
            out, info, _, _ = loglike_grad(Xd, yd, e2, desc, work=work)
        else:
            out, info, _, _ = loglike_grad(banded[0], banded[1], banded[2], desc, work=work, row_end=banded[3])
            self.n_banded_evaluations = getattr(self, "n_banded_evaluations", 0) + 1
        self.n_evaluations += 1
        o = out.cpu().numpy()
        if o[0] != o[0]:
            from ._cabi import TgpError
            raise TgpError("tgp_loglike_grad: internal synchronisation timed out (info = %d)" % int(info.item()))
        return float(o[0]), J.T @ o[3:3 + J.shape[0]]

    @staticmethod
    def _value_and_fd_gradient(fun, rank, world):
        """f(theta) and its forward-difference gradient with the n_theta + 1 probes dealt round-robin to the
        ranks (probe i on rank i % world) and combined with one all-reduce."""
        import torch
        import torch.distributed as tdist

        on_gpu = tdist.get_backend() == "nccl"

        def value_and_grad(theta):
            theta = np.asarray(theta, dtype=float)
            probes = [theta] + [theta + _FD_STEP * np.eye(len(theta))[i] for i in range(len(theta))]
            vals = torch.zeros(len(probes), dtype=torch.float64)
            for i, p in enumerate(probes):
                if i % world == rank:
                    v = fun(p)
                    vals[i] = v if np.isfinite(v) else 1e300  # keep the all-reduce finite; mapped back below
            if on_gpu:
                vals = vals.cuda()
            tdist.all_reduce(vals)
            vals = vals.cpu().numpy()
            vals = np.where(vals >= 1e300, np.inf, vals)
            return float(vals[0]), (vals[1:] - vals[0]) / _FD_STEP

        return value_and_grad

    def optimizer(self, kernel):
        """Maximise the likelihood over theta starting from `kernel.theta` (scipy L-BFGS-B, no bounds,
        forward-difference gradient, or the analytic one when ANALYTIC_GRADIENT is set) and return the fitted kernel;
        keeps `_kernel` and `_logL`."""

        def minus_logl(theta):
            return -self.log_likelihood(kernel.clone_with_theta(theta))

        import os
        from . import dist

        rank, world = dist.rank_world(None)
        if self.ANALYTIC_GRADIENT:
            def minus_logl_and_grad(theta):
                v, g = self.log_likelihood_and_gradient(kernel.clone_with_theta(theta))
                return -v, -g

            best = optimize.minimize(minus_logl_and_grad, kernel.theta, method="L-BFGS-B", jac=True)["x"]
        elif world > 1 and (DISTRIBUTED_FD or os.environ.get("TREEGP_B200_DIST_FD") == "1"):
            best = optimize.minimize(self._value_and_fd_gradient(minus_logl, rank, world), kernel.theta,
                                     method="L-BFGS-B", jac=True)["x"]
        else:
            # unbounded L-BFGS-B with scipy's forward-difference gradient, as log_likelihood.py:56-57
            best = optimize.minimize(minus_logl, kernel.theta, method="L-BFGS-B")["x"]
        kernel = kernel.clone_with_theta(best)
        self._kernel = copy.deepcopy(kernel)
        self._logL = self.log_likelihood(self._kernel)
        return kernel
