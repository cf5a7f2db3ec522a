"""GPInterpolation: Gaussian-process interpolation of a single surface, solved on the B200.

Host-side mirror of /root/reference/treegp/gp_interp.py:15-291 -- same constructor keywords and
defaults (:54-67), ``initialize`` (:196), ``solve`` (:245), ``predict`` (:143), ``return_2pcf``
(:260), ``return_log_likelihood`` (:277), same error behaviour (TypeError for a non-string kernel
:84-89, ValueError for an unknown optimizer :91-95) and the same private attribute names that the
reference's tests read (``kernel_template``, ``kernel``, ``_optimizer``, ``_alpha``, ``_mean``...).

What changed is the arithmetic: ``return_gp_predict`` (:168-194) is K build -> DMMA Cholesky ->
triangular sweeps -> fused K(X*,X).alpha on the device through the C ABI; the factor and alpha are
cached on the device between predicts exactly where the reference caches ``_alpha``.  The covariance
is computed from ONE factorisation as K** - V V^T with V = K* L^-T (the reference's second
``cholesky`` of an overwritten buffer is a latent bug under scipy >= 1.15, SURVEY.md section 4.3).
"""
import copy

import numpy as np

from . import _cabi, backend
from .kernels import eval_kernel, lower
from .log_likelihood import log_likelihood
from .two_pcf import two_pcf


class GPInterpolation(object):
    """Gaussian-process interpolation of one scalar surface sampled at scattered 1-D or 2-D positions.

    Several outputs (extension): a y of shape (n, r), 1 <= r <= 8, holds r fields measured at the same points with
    the same errors.  They are interpolated as r independent GPs sharing one kernel (scikit-learn's
    GaussianProcessRegressor with multi-target y): one factorisation serves all of them, predictions are (m, r), the
    log-likelihood is the sum over the outputs and "log-likelihood" fits the shared kernel to all of them together.

    Constructor keywords (names, order and defaults as in the reference):

    kernel          kernel string, evaluated by `eval_kernel` (e.g. "4.0 * AnisotropicRBF(invLam=array(...))")
    optimizer       "none" keeps the kernel as given; "two-pcf" / "anisotropic" fit it to the isotropic /
                    two-dimensional 2-point correlation function; "log-likelihood" maximises the marginal
                    likelihood
    normalize       subtract the mean of the (mean-function-subtracted) data before solving
    p0              start [size, g1, g2] of the robust anisotropic fit
    white_noise     extra uncorrelated noise, added in quadrature to y_err
    n_neighbors     neighbours averaged when looking up the mean function (average_fits only)
    average_fits    FITS table written by `meanify` holding the mean function; indice_meanify picks a column
    nbins           bins of the 1-D correlation function, or bins per axis of the 2-D one
    min_sep,max_sep separation range of the correlation function (defaults chosen from the data)
    """

    def __init__(
        self,
        kernel="RBF(1)",
        optimizer="two-pcf",
        normalize=True,
        p0=[3000.0, 0.0, 0.0],
        white_noise=0.0,
        n_neighbors=4,
        average_fits=None,
        indice_meanify=None,
        nbins=20,
        min_sep=None,
        max_sep=None,
    ):
        self.normalize = normalize
        self.optimizer = optimizer
        self.white_noise = white_noise
        self.n_neighbors = n_neighbors
        self.nbins = nbins
        self.min_sep = min_sep
        self.max_sep = max_sep
        self.robust_fit = self.optimizer == "anisotropic"
        self.p0_robust_fit = p0
        self.indice_meanify = indice_meanify

        if not isinstance(kernel, str):
            raise TypeError("kernel should be a string a list or a numpy.ndarray of string")
        self.kernel_template = eval_kernel(kernel)

        if self.optimizer not in ["anisotropic", "two-pcf", "log-likelihood", "none"]:
            raise ValueError(
                "Only anisotropic, two-pcf, log-likelihood and none are supported for optimizer. "
                "Current value: %s" % (self.optimizer)
            )

        if average_fits is not None:
            from .meanify import read_average

            X0, y0 = read_average(average_fits)
        else:
            X0, y0 = None, None
        self._X0 = X0
        self._y0 = y0
        self._has_average = average_fits is not None
        self._alpha = None
        self._factor = None

    # ---------------------------------------------------------------------------------------
    def _fit(self, kernel, X, y, y_err):
        """Run the configured optimizer on (X, y, y_err) and return the fitted kernel (gp_interp.py:111-141)."""
        self._alpha = None
        self._factor = None
        if self.optimizer in ["two-pcf", "anisotropic"]:
            self._optimizer = two_pcf(
                X,
                y,
                y_err,
                self.min_sep,
                self.max_sep,
                nbins=self.nbins,
                anisotropic=self.optimizer == "anisotropic",
                robust_fit=self.robust_fit,
                p0=self.p0_robust_fit,
            )
            kernel = self._optimizer.optimizer(kernel)
        elif self.optimizer == "log-likelihood":
            self._optimizer = log_likelihood(X, y, y_err)
            kernel = self._optimizer.optimizer(kernel)
        return kernel

    def predict(self, X, return_cov=False):
        """Posterior mean at the positions X (m, 1|2), plus the full (m, m) posterior covariance when
        return_cov is set (gp_interp.py:143-166)."""
        y_interp, y_cov = self.return_gp_predict(
            self._y - self._mean - self._spatial_average,
            self._X,
            X,
            self.kernel,
            y_err=self._y_err,
            return_cov=return_cov,
        )
        y_interp = y_interp + self._mean + self._build_average_meanify(X)
        if return_cov:
            return y_interp, y_cov
        return y_interp

    # K + diag(y_err^2) is factorised inside its envelope when the kernel's support is short against the field
    # (backend.plan_envelope); False: always the dense factorisation
    BANDED_SOLVE = True
    _envelope = None

    # predict_var: solve only the trailing sub-system that a chunk of neighbouring test points can be correlated with
    # (backend.predict_var_windowed) whenever that is cheaper than the plain solves on the cached factor
    WINDOWED_VARIANCE = True
    VAR_CHUNK = None   # test points per pass (None: a workspace of about 2 GiB)

    def predict_var(self, X):
        """Extension (not in the reference): mean and DIAGONAL predictive variance for any number of
        test points -- what the reference's callers take from ``np.diag(y_cov)``, without the M x M
        matrix (8 TB at M = 1e6)."""
        self._ensure_solved(self._y - self._mean - self._spatial_average, self._X, self.kernel, self._y_err)
        Xd, desc, ws = self._factor
        Xs = backend.as_points(X)
        mean = backend.predict_mean(Xs, Xd, desc, self._alpha_dev)
        var, self._var_plan = None, {}
        if self.WINDOWED_VARIANCE:
            var = backend.predict_var_windowed(Xs, Xd, desc, self._e2_dev, chunk=self.VAR_CHUNK, stats=self._var_plan)
        if var is None:
            var = backend.predict_var(Xs, Xd, desc, ws, chunk=self.VAR_CHUNK,
                                      row_end=None if self._envelope is None else self._envelope["row_end"])
        y = mean.cpu().numpy() + self._mean + self._build_average_meanify(X)
        return y, var.cpu().numpy()

    def _solve(self, Xd, yd, e2, desc):
        """K + diag(e2) -> L -> alpha = K^-1 y on the device for y (n,) or (n, r).  A kernel whose support is short
        against the field: with the points sorted along one axis K is zero (below 1e-40 amp) outside an envelope that
        its Cholesky factor keeps -- factorise inside it (N bw^2 flop instead of N^3 / 3); X, y_err^2, alpha and the
        factor are then in the sorted order.  Returns (X, y_err^2, alpha, workspace holding L, envelope plan or None);
        raises as scipy.linalg.cholesky does (gp_interp.py:181) when K is not positive definite."""
        env = backend.plan_envelope(Xd, desc) if self.BANDED_SOLVE else None
        if env is not None:
            Xd, yd, e2 = Xd[env["order"]].contiguous(), yd[env["order"]].contiguous(), e2[env["order"]].contiguous()
        # one call: K (lower) -> L with y riding through the factorisation as extra rows (forward substitution
        # for free), then the backward sweep (want_alpha)
        _, info, alpha, ws = backend.loglike(Xd, yd, e2, desc, want_alpha=True,
                                             row_end=None if env is None else env["row_end"])
        bad = int(info.item())
        if bad < 0:
            raise _cabi.TgpError("tgp_loglike: internal synchronisation timed out (info = %d)" % bad)
        if bad != 0:
            raise np.linalg.LinAlgError("%d-th leading minor of the array is not positive definite" % bad)
        return Xd, e2, alpha, ws, env

    def _ensure_solved(self, y, X1, kernel, y_err):
        """K + diag(y_err^2) -> L -> alpha on the device, cached like ``_alpha`` (gp_interp.py:179-182).  A y of
        shape (n, r) gives alpha (n, r) from the same factorisation.  With an envelope the factor, X and alpha are held
        in the sorted order; `_alpha` (host) in the caller's."""
        if self._alpha is not None and self._factor is not None:
            return
        Xd = backend.as_points(X1)
        desc = lower(kernel, Xd.shape[1])
        e2 = backend.to_device(np.asarray(y_err, dtype=np.float64).reshape(-1) ** 2)
        Xd, e2, alpha, ws, env = self._solve(Xd, _device_outputs(y), e2, desc)
        self._factor = (Xd, desc, ws)
        self._e2_dev = e2        # y_err^2 in the order of Xd
        self._envelope = env
        self._alpha_dev = alpha
        self._alpha = (alpha if env is None else _unsort(alpha, env["order"])).cpu().numpy()

    def loo_predict(self):
        """Extension (not in the reference): leave-one-out predictions at every training point, in the caller's
        order, without refitting -- (mean, var) with mean_i = y_i - alpha_i / Z_ii and var_i = 1 / Z_ii - y_err_i^2,
        Z = (K + diag(y_err^2))^-1 (its diagonal from the selected inverse, tgp_selinv), y_err after the white noise.
        This is what predict / predict_var return at X_i from the other N - 1 points with the same kernel; the
        normalising mean and the mean function keep their all-point values and are added back as predict does.
        Factorises into a workspace of its own: the cached factor of predict_var / return_cov stays as it is.
        Several outputs: mean (n, r) with mean_ic = y_ic - alpha_ic / Z_ii, var (n,) shared by the outputs."""
        y = np.asarray(self._y - self._mean - self._spatial_average, dtype=np.float64)
        multi = y.ndim == 2
        if not multi:
            y = y.reshape(-1)
        Xd = backend.as_points(self._X)
        n = Xd.shape[0]
        desc = lower(self.kernel, Xd.shape[1])
        e2_host = np.asarray(self._y_err, dtype=np.float64).reshape(-1) ** 2
        _, _, alpha, ws, env = self._solve(Xd, backend.to_device(y), backend.to_device(e2_host), desc)
        backend.selinv(ws, n, row_end=None if env is None else env["row_end"])
        zdiag = ws[:, :n].diagonal()
        if env is not None:
            alpha, zdiag = _unsort(alpha, env["order"]), _unsort(zdiag, env["order"])
        alpha, zdiag = alpha.cpu().numpy(), zdiag.cpu().numpy()
        mean = y - alpha / (zdiag[:, None] if multi else zdiag) + self._mean + self._spatial_average
        return mean, 1.0 / zdiag - e2_host

    def return_gp_predict(self, y, X1, X2, kernel, y_err, return_cov=False):
        """GP algebra for residuals y at X1 with errors y_err, evaluated at X2 with `kernel`
        (gp_interp.py:168-194): returns (mean, covariance-or-None)."""
        self._ensure_solved(y, X1, kernel, y_err)
        Xd, desc, ws = self._factor
        n = Xd.shape[0]
        Xs = backend.as_points(X2)
        m = Xs.shape[0]
        y_predict = backend.predict_mean(Xs, Xd, desc, self._alpha_dev).cpu().numpy()
        if not return_cov:
            return y_predict, None
        # y_cov = K** - K* (K + s^2 I)^-1 K*^T = K** - V V^T,  V = K* L^-T  (gp_interp.py:187-191)
        V = backend.kmat_cross(Xs, Xd, desc)
        backend.trsm_rows(ws, n, V, m, row_end=None if self._envelope is None else self._envelope["row_end"])
        cov = backend.kmat_sym(Xs, desc)
        backend.gemm_nt_sub(cov, m, m, V, V, n)
        return y_predict, cov[:, :m].cpu().numpy()

    def initialize(self, X, y, y_err=None):
        """Attach the data: positions X (n, 1|2), values y (n,), optional errors y_err (n,); looks up the
        mean function, folds in the white noise, computes the normalising mean and drops any cached
        solve (gp_interp.py:196-227)."""
        multi = np.ndim(y) == 2
        if multi:
            _check_multi_inputs(y, y_err, self._has_average, self._y0, self.indice_meanify)
        self.kernel = copy.deepcopy(self.kernel_template)
        self._X = X
        self._y = y
        if y_err is None:
            y_err = np.zeros(len(y)) if multi else np.zeros_like(y)
        self._y_err = y_err

        if self._X0 is None:
            self._X0 = np.zeros_like(self._X)
            self._y0 = np.zeros_like(self._y)
        self._spatial_average = self._build_average_meanify(X)

        if self.white_noise > 0:
            y_err = np.sqrt(np.array(self._y_err, dtype=float) ** 2 + self.white_noise ** 2)
        self._y_err = y_err

        if self.normalize:
            # several outputs: one mean per column, _mean has shape (r,); column by column, so that each output is
            # normalised exactly as it would be on its own (numpy sums a strided axis in another order)
            if multi:
                res = np.asarray(y - self._spatial_average)
                self._mean = np.array([np.mean(np.ascontiguousarray(res[:, c])) for c in range(res.shape[1])])
            else:
                self._mean = np.mean(y - self._spatial_average)
        else:
            self._mean = 0.0
        # alpha / L are recomputed whenever the input data change
        self._alpha = None
        self._factor = None

    def _build_average_meanify(self, X):
        """Mean function at X: uniform mean of the `n_neighbors` nearest grid values of the meanify table,
        or zeros when no table was given (gp_interp.py:229-243)."""
        X = np.asarray(X)
        multi = np.ndim(self._y) == 2
        if np.count_nonzero(self._X0) == 0:
            return np.zeros((len(X[:, 0]), np.shape(self._y)[1])) if multi else np.zeros(len(X[:, 0]))
        from .meanify import knn_average

        average = knn_average(self._X0, self._y0, X, self.n_neighbors)
        if self.indice_meanify is not None:
            average = average[:, list(self.indice_meanify) if multi else self.indice_meanify]
        return average

    def solve(self):
        """Fit the kernel hyper-parameters with the configured optimizer (gp_interp.py:245-258)."""
        self._check_2pcf_output()
        self._init_theta = [copy.deepcopy(self.kernel).theta]
        self.kernel = self._fit(
            self.kernel,
            self._X,
            self._y - self._mean - self._spatial_average,
            self._y_err,
        )

    def return_2pcf(self):
        """xi, its weight matrix, separations, bin coordinates and mask for the current data
        (gp_interp.py:260-275)."""
        self._check_2pcf_output(always=True)
        pcf = two_pcf(
            self._X,
            self._y - self._mean - self._spatial_average,
            self._y_err,
            self.min_sep,
            self.max_sep,
            nbins=self.nbins,
            anisotropic=self.optimizer == "anisotropic",
        )
        return pcf.return_2pcf()

    def _check_2pcf_output(self, always=False):
        """The 2-point correlation function fit is defined for one scalar field."""
        if np.ndim(self._y) == 2 and (always or self.optimizer in ["two-pcf", "anisotropic"]):
            raise ValueError(TWO_PCF_NEEDS_1D_Y)

    def return_log_likelihood(self, theta=None):
        """Marginal log-likelihood of the current data for the current kernel, or for `theta` if given
        (gp_interp.py:277-291)."""
        kernel = copy.deepcopy(self.kernel)
        if theta is not None:
            kernel = kernel.clone_with_theta(theta)
        logl = log_likelihood(self._X, self._y - self._mean - self._spatial_average, self._y_err)
        return logl.log_likelihood(kernel)

    def plot_fitted_kernel(self):
        """Figure with the measured 2-D 2-point correlation function, the fitted kernel and their
        difference (gp_interp.py:293-377).  Host-only; needs matplotlib (imported lazily, as in the
        reference -- an ImportError surfaces if it is not installed)."""
        if self.optimizer in ["none", "log-likehood", "two-pcf"]:
            raise NotImplementedError("This method is only available for anisotropic optimizer")
        import os

        if os.getenv("GITHUB_ACTIONS") == "true":
            import matplotlib

            matplotlib.use("Agg")
        import matplotlib.pyplot as plt

        opt = self._optimizer
        lag = opt._2pcf_dist
        extent = [lag[:, 0].min(), lag[:, 0].max(), lag[:, 1].min(), lag[:, 1].max()]
        n = int(np.sqrt(len(opt._2pcf)))
        vmax = np.max(opt._2pcf)
        panels = [(opt._2pcf.reshape(n, n), "Measured 2-PCF", "$\\xi$"),
                  (opt._2pcf_fit.reshape(n, n), "Fitted 2-PCF", "$\\xi'$"),
                  (opt._2pcf.reshape(n, n) - opt._2pcf_fit.reshape(n, n), "Difference", "$\\xi - \\xi'$")]
        fig = plt.figure(figsize=(14, 4))
        plt.subplots_adjust(wspace=0.5, left=0.07, right=0.95, bottom=0.1, top=0.92)
        for i, (img, title, label) in enumerate(panels, start=1):
            plt.subplot(1, 3, i)
            plt.imshow(img, extent=extent, interpolation="nearest", origin="lower", vmin=-vmax, vmax=vmax,
                       cmap=plt.cm.seismic)
            cbar = plt.colorbar()
            cbar.formatter.set_powerlimits((0, 0))
            cbar.update_ticks()
            cbar.set_label(label, fontsize=16)
            plt.xlabel(r"$\Delta x$", fontsize=16)
            if i == 1:
                plt.ylabel(r"$\Delta y$", fontsize=16)
            plt.title(title, fontsize=16)
        return fig


# the 2-point correlation function fit is defined for one scalar field (GPInterpolation and GPInterpolationBatch)
TWO_PCF_NEEDS_1D_Y = ("the two-pcf / anisotropic fit and return_2pcf need a 1-D y; with several outputs use "
                      "optimizer='log-likelihood' or 'none'")


def _unsort(t, order):
    """The rows of t, which are in the order `order` of the caller's rows, back in the caller's order."""
    u = t.new_empty(t.shape)
    u[order] = t
    return u


def _device_outputs(y):
    """y on the device: (n,) for one output (any shape flattened, as the reference does), (n, r) for several."""
    y = np.asarray(y, dtype=np.float64)
    return backend.to_device(y if y.ndim == 2 else y.reshape(-1))


def _check_multi_inputs(y, y_err, has_average, y0, indice_meanify):
    """Several outputs: y (n, r) with 1 <= r <= TGP_MAX_RHS, y_err None or (n,) shared by the outputs, and with a
    meanify table r column indices (None only when the table has exactly r columns)."""
    n, r = np.shape(y)
    if not 1 <= r <= _cabi.MAX_RHS:
        raise ValueError("y has %d outputs; at most %d (TGP_MAX_RHS) share one kernel" % (r, _cabi.MAX_RHS))
    if y_err is not None and np.shape(y_err) != (n,):
        raise ValueError("with several outputs y_err must have shape (n,) = (%d,), shared by the outputs; got %r"
                         % (n, np.shape(y_err)))
    if has_average:
        ncols = np.shape(y0)[1] if np.ndim(y0) == 2 else 1
        if indice_meanify is None:
            if np.ndim(y0) != 2 or ncols != r:
                raise ValueError("indice_meanify=None needs a meanify table with exactly %d columns; it has %d"
                                 % (r, ncols))
        else:
            idx = np.atleast_1d(np.asarray(indice_meanify))
            if (idx.ndim != 1 or len(idx) != r or idx.dtype.kind not in "iu" or np.ndim(y0) != 2
                    or np.any(idx < -ncols) or np.any(idx >= ncols)):
                raise ValueError("indice_meanify must list %d column indices of the meanify table (%d columns); got %r"
                                 % (r, ncols, indice_meanify))
