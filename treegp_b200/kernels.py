"""Covariance functions with the scikit-learn ``Kernel`` protocol, evaluated on the B200.

Host-side mirror of /root/reference/treegp/kernels.py: the same public names (``eval_kernel``,
``AnisotropicRBF``, ``VonKarman``, ``AnisotropicVonKarman``), constructor arguments, ``theta``
parameterisation (log-Cholesky of the inverse metric, kernels.py:163-179 / :397-413) and ``bounds``,
so kernel strings such as ``"4.0 * AnisotropicRBF(invLam=array([[...]]))"`` keep working.  What
changes is where the numbers come from: ``__call__`` lowers the kernel to the POD descriptor of
include/treegp_b200.h and runs the tiled CUDA build (csrc/kmat.cu) instead of
pdist/cdist + scipy.special.kv.

``lower_kernel`` is the bridge used by GPInterpolation / log_likelihood / two_pcf to keep whole
solves on the device; ``lower_kernel_sum`` lowers sums of such terms plus a ``WhiteKernel`` level, and ``lower``
picks whichever of the two applies.
"""
import numpy as np
from sklearn.gaussian_process import kernels as _skk
from sklearn.gaussian_process.kernels import (
    ConstantKernel,
    Hyperparameter,
    Kernel,
    Matern,
    NormalizedKernelMixin,
    Product,
    RBF,
    StationaryKernelMixin,
    Sum,
    WhiteKernel,
)

from . import _cabi
from ._cabi import TgpKernel, TgpKernelSum

__all__ = ["eval_kernel", "AnisotropicRBF", "VonKarman", "AnisotropicVonKarman", "lower_kernel",
           "lower_kernel_jacobian", "lower_kernel_sum", "lower_kernel_sum_jacobian", "lower", "lower_jacobian"]


# ------------------------------------------------------------------------------------------------
# device evaluation shared by the three kernels
# ------------------------------------------------------------------------------------------------
def _device_call(desc, X, Y):
    """Evaluate amp * f on the GPU and return a numpy array, (N, N) or (N, M)."""
    from . import backend

    X = np.atleast_2d(np.asarray(X, dtype=np.float64))
    if Y is None:
        n = X.shape[0]
        out = backend.kmat_sym(X, desc)
        return out[:, :n].cpu().numpy()
    Y = np.atleast_2d(np.asarray(Y, dtype=np.float64))
    out = backend.kmat_cross(X, Y, desc)
    return out[:, : Y.shape[0]].cpu().numpy()


def _descriptor(family, ndim, amp, metric):
    m = np.asarray(metric, dtype=np.float64)
    if ndim == 1:
        return TgpKernel(family, 1, float(amp), float(m[0, 0]), 0.0, 0.0)
    if ndim != 2:
        raise _cabi.TgpError("the B200 backend handles 1-D and 2-D coordinates; got ndim=%d" % ndim)
    if abs(m[0, 1] - m[1, 0]) > 1e-12 * max(1.0, abs(m[0, 1])):
        raise ValueError("inverse metric must be symmetric")
    return TgpKernel(family, 2, float(amp), float(m[0, 0]), float(0.5 * (m[0, 1] + m[1, 0])), float(m[1, 1]))


# ------------------------------------------------------------------------------------------------
# kernels parameterised by a full inverse metric
# ------------------------------------------------------------------------------------------------
class _MetricKernel(StationaryKernelMixin, NormalizedKernelMixin, Kernel):
    """Stationary kernel k(x, y) = f((x-y)^T invLam (x-y)) with theta = log-Cholesky(invLam).

    theta[:n] are the logs of the diagonal of L, theta[n:] its strict lower triangle (row-major),
    invLam = L L^T -- the unconstrained parameterisation of kernels.py:71-83.
    """

    _family = None

    def __init__(self, invLam=None, scale_length=None, bounds=(-5, 5)):
        if scale_length is not None:
            if invLam is not None:
                raise TypeError("Cannot set both invLam and scale_length in %s." % type(self).__name__)
            invLam = np.diag(1.0 / np.array(scale_length) ** 2)
        if invLam is None:
            raise TypeError("Exactly one of invLam and scale_length must be provided.")
        self.ndim = invLam.shape[0]
        self.ntheta = self.ndim * (self.ndim + 1) // 2
        self._d = np.diag_indices(self.ndim)
        self._t = np.tril_indices(self.ndim, -1)
        self.set_params(invLam)
        b = np.array(bounds)
        if b.ndim == 1:
            b = np.tile(b, (self.ntheta, 1))
        assert b.shape == (self.ntheta, 2)
        self._bounds = b

    # -- sklearn plumbing ---------------------------------------------------------------------
    @property
    def hyperparameter_cholesky_factor(self):
        return Hyperparameter("CholeskyFactor", "numeric", (1e-5, 1e5), int(self.ntheta))

    def get_params(self, deep=True):
        return {"invLam": self.invLam}

    def set_params(self, invLam=None):
        if invLam is None:
            return
        self.invLam = invLam
        self._L = np.linalg.cholesky(self.invLam)
        self._theta = np.concatenate([np.log(self._L[self._d]), self._L[self._t]])

    @property
    def theta(self):
        return self._theta

    @theta.setter
    def theta(self, theta):
        theta = np.asarray(theta, dtype=float)
        L = np.zeros((self.ndim, self.ndim))
        L[self._d] = np.exp(theta[: self.ndim])
        L[self._t] = theta[self.ndim:]
        self._theta = theta
        self._L = L
        self.invLam = L @ L.T

    @property
    def bounds(self):
        return self._bounds

    def __repr__(self):
        return "{0}(invLam={1!r})".format(type(self).__name__, self.invLam)

    # -- evaluation ---------------------------------------------------------------------------
    def descriptor(self, amp=1.0):
        return _descriptor(self._family, self.ndim, amp, self.invLam)

    def __call__(self, X, Y=None, eval_gradient=False):
        if eval_gradient:
            return self._with_gradient(X, Y)
        return _device_call(self.descriptor(), X, Y)

    def _with_gradient(self, X, Y):
        raise ValueError("Gradient can not be evaluated.")


class AnisotropicRBF(_MetricKernel):
    """Squared-exponential kernel with an arbitrary inverse covariance:
    k = exp(-1/2 (x-y)^T invLam (x-y)).  Mirror of kernels.py:62-186.

    :param invLam:        inverse covariance matrix (exactly one of invLam / scale_length).
    :param scale_length:  per-axis scale lengths; invLam = diag(1 / scale_length^2).
    :param bounds:        bounds on theta, a pair or an (ntheta, 2) array.
    """

    _family = _cabi.FAM_RBF

    def _with_gradient(self, X, Y):
        # dK/dtheta_k = -1/2 K * (dx^T dInvLam/dtheta_k dx)   (kernels.py:128-150).  Not on the hot
        # path (log_likelihood.py:57 passes no jac): K comes from the device, the contraction with
        # the ntheta small matrices is done on the host.
        if Y is not None:
            raise ValueError("Gradient can only be evaluated when Y is None.")
        X = np.atleast_2d(np.asarray(X, dtype=np.float64))
        K = _device_call(self.descriptor(), X, None)
        n, nth = self.ndim, self.ntheta
        dL = np.zeros((nth, n, n))
        for a in range(n):
            dL[a, a, a] = self._L[a, a]
        for a, (i, j) in enumerate(zip(*self._t)):
            dL[n + a, i, j] = 1.0
        half = dL @ self._L.T
        dM = half + np.transpose(half, (0, 2, 1))
        dX = X[:, None, :] - X[None, :, :]
        quad = np.einsum("pqi,kij,pqj->pqk", dX, dM, dX)
        return K, -0.5 * K[:, :, None] * quad


class AnisotropicVonKarman(_MetricKernel):
    """von Karman (Kolmogorov-turbulence) correlation with an arbitrary inverse covariance:
    k = d^(5/6) K_{5/6}(2 pi d) / lim0 with d the Mahalanobis distance.  Mirror of kernels.py:304-420.
    """

    _family = _cabi.FAM_VONKARMAN


# ------------------------------------------------------------------------------------------------
# isotropic von Karman with a length scale
# ------------------------------------------------------------------------------------------------
class VonKarman(StationaryKernelMixin, NormalizedKernelMixin, Kernel):
    """k = (r/l)^(5/6) K_{5/6}(2 pi r / l) / lim0.  Mirror of kernels.py:189-301.

    :param length_scale:         float (isotropic) -- an array of per-axis scales is accepted for
                                 scalar-equivalent shapes as in sklearn.
    :param length_scale_bounds:  bounds on length_scale.
    """

    def __init__(self, length_scale=1.0, length_scale_bounds=(1e-5, 1e5)):
        self.length_scale = length_scale
        self.length_scale_bounds = length_scale_bounds

    @property
    def anisotropic(self):
        return np.iterable(self.length_scale) and len(self.length_scale) > 1

    @property
    def hyperparameter_length_scale(self):
        if self.anisotropic:
            return Hyperparameter("length_scale", "numeric", self.length_scale_bounds, len(self.length_scale))
        return Hyperparameter("length_scale", "numeric", self.length_scale_bounds)

    def descriptor(self, ndim, amp=1.0):
        ls = np.ravel(np.asarray(self.length_scale, dtype=float))
        if ls.size == 1:
            ls = np.repeat(ls, ndim)
        if ls.size != ndim:
            raise ValueError("length_scale has %d entries for %d-D coordinates" % (ls.size, ndim))
        return _descriptor(_cabi.FAM_VONKARMAN, ndim, amp, np.diag(1.0 / ls ** 2))

    def __call__(self, X, Y=None, eval_gradient=False):
        X = np.atleast_2d(np.asarray(X, dtype=np.float64))
        K = _device_call(self.descriptor(X.shape[1]), X, Y)
        if not eval_gradient:
            return K
        if Y is not None:
            raise ValueError("Gradient can only be evaluated when Y is None.")
        if self.hyperparameter_length_scale.fixed:
            return K, np.empty((X.shape[0], X.shape[0], 0))
        if self.anisotropic:
            raise ValueError("Gradient can only be evaluated with isotropic VonKarman kernel for the moment.")
        # the reference's (approximate) expression K * r  (kernels.py:283-285)
        r = np.sqrt(((X[:, None, :] - X[None, :, :]) ** 2).sum(-1))
        return K, (K * r)[:, :, None]

    def __repr__(self):
        if self.anisotropic:
            return "{0}(length_scale=[{1}])".format(
                type(self).__name__, ", ".join("{0:.3g}".format(v) for v in self.length_scale))
        return "{0}(length_scale={1:.3g})".format(type(self).__name__, np.ravel(self.length_scale)[0])


# ------------------------------------------------------------------------------------------------
# kernel strings
# ------------------------------------------------------------------------------------------------
def _kernel_namespace():
    ns = {}
    stack = list(Kernel.__subclasses__())
    while stack:
        cls = stack.pop()
        ns.setdefault(cls.__name__, cls)
        stack.extend(cls.__subclasses__())
    for name in dir(_skk):
        obj = getattr(_skk, name)
        if isinstance(obj, type) and issubclass(obj, Kernel):
            ns.setdefault(name, obj)
    ns["array"] = np.array
    return ns


def eval_kernel(kernel):
    """Turn a kernel string (a sklearn / treegp kernel ``repr`` or any expression over them, e.g.
    ``"2.0**2 * RBF(0.5)"``) into a kernel object.  Mirror of kernels.py:17-59: every subclass of
    sklearn's ``Kernel`` plus numpy's ``array`` is in scope."""
    try:
        k = eval(kernel, _kernel_namespace())
    except Exception as e:
        raise RuntimeError("Failed to evaluate kernel string {0!r}.  Original exception: {1}".format(kernel, e))
    if isinstance(getattr(k, "theta", None), property) or not isinstance(k, Kernel):
        raise TypeError("String provided was not initialized properly")
    return k


# ------------------------------------------------------------------------------------------------
# lowering sklearn kernel trees to the device descriptor
# ------------------------------------------------------------------------------------------------
def _iso_metric(length_scale, ndim, what):
    ls = np.ravel(np.asarray(length_scale, dtype=float))
    if ls.size == 1:
        ls = np.repeat(ls, ndim)
    if ls.size != ndim:
        raise ValueError("%s length_scale has %d entries for %d-D coordinates" % (what, ls.size, ndim))
    return np.diag(1.0 / ls ** 2)


def lower_kernel(kernel, ndim):
    """sklearn kernel tree -> ``TgpKernel``.

    Supported: an optional product with any number of ``ConstantKernel`` factors around one of
    RBF, Matern(nu in {0.5, 1.5, 2.5, inf}), VonKarman, AnisotropicRBF, AnisotropicVonKarman --
    the surface the reference's tests, docs and notebooks exercise (SURVEY.md section 3.5).  Anything
    else raises: there is no CPU fallback to silently take over.
    """
    amp = 1.0
    base = None
    stack = [kernel]
    while stack:
        k = stack.pop()
        if isinstance(k, Product):
            stack.extend([k.k1, k.k2])
        elif isinstance(k, ConstantKernel):
            amp *= float(k.constant_value)
        elif base is None:
            base = k
        else:
            raise _cabi.TgpError("unsupported kernel for the B200 backend (more than one non-constant factor): %r"
                                 % (kernel,))
    if base is None:
        raise _cabi.TgpError("unsupported kernel for the B200 backend (no stationary factor): %r" % (kernel,))
    if isinstance(base, _MetricKernel):
        if base.ndim != ndim:
            raise ValueError("kernel is %d-D but coordinates are %d-D" % (base.ndim, ndim))
        return base.descriptor(amp)
    if isinstance(base, VonKarman):
        return base.descriptor(ndim, amp)
    if isinstance(base, Matern):  # Matern subclasses RBF: test it first
        fam = {0.5: _cabi.FAM_MATERN12, 1.5: _cabi.FAM_MATERN32, 2.5: _cabi.FAM_MATERN52,
               np.inf: _cabi.FAM_RBF}.get(float(base.nu))
        if fam is None:
            raise _cabi.TgpError("Matern(nu=%r) is not supported by the B200 backend (nu in 0.5, 1.5, 2.5, inf)"
                                 % (base.nu,))
        return _descriptor(fam, ndim, amp, _iso_metric(base.length_scale, ndim, "Matern"))
    if isinstance(base, RBF):
        return _descriptor(_cabi.FAM_RBF, ndim, amp, _iso_metric(base.length_scale, ndim, "RBF"))
    raise _cabi.TgpError("unsupported kernel for the B200 backend: %r" % (kernel,))


def _metric_columns(dM, ndim):
    """Symmetric 2 x 2 (or 1 x 1) derivative of the inverse metric -> rows (m00, m01, m11) of the Jacobian."""
    dM = np.atleast_2d(dM)
    if ndim == 1:
        return np.array([dM[0, 0], 0.0, 0.0])
    return np.array([dM[0, 0], dM[0, 1], dM[1, 1]])


def _factor_jacobian(k, ndim):
    """Columns d(ln a, m00, m01, m11) / d theta_k of one factor of the product, in the order of k.theta."""
    if isinstance(k, ConstantKernel):
        return [] if k.hyperparameter_constant_value.fixed else [np.array([1.0, 0.0, 0.0, 0.0])]
    if isinstance(k, _MetricKernel):
        if k.ndim != ndim:
            raise ValueError("kernel is %d-D but coordinates are %d-D" % (k.ndim, ndim))
        n, L = k.ndim, k._L
        cols = []
        for a in range(n):                                  # theta[a] = ln L[a, a]
            dL = np.zeros((n, n))
            dL[a, a] = L[a, a]
            cols.append(dL)
        for i, j in zip(*k._t):                             # theta[n + ...] = L[i, j], i > j
            dL = np.zeros((n, n))
            dL[i, j] = 1.0
            cols.append(dL)
        return [np.concatenate([[0.0], _metric_columns(dL @ L.T + L @ dL.T, ndim)]) for dL in cols]
    if isinstance(k, (VonKarman, RBF)):   # Matern subclasses RBF; its nu is not a hyper-parameter
        if k.hyperparameter_length_scale.fixed:
            return []
        ls = np.ravel(np.asarray(k.length_scale, dtype=float))
        if ls.size == 1:   # one theta: d M / d ln l = -2 l^-2 I
            return [np.concatenate([[0.0], _metric_columns(-2.0 * np.eye(ndim) / ls[0] ** 2, ndim)])]
        if ls.size != ndim:
            raise ValueError("length_scale has %d entries for %d-D coordinates" % (ls.size, ndim))
        cols = []
        for a in range(ndim):   # d M / d ln l_a = -2 l_a^-2 e_a e_a^T
            dM = np.zeros((ndim, ndim))
            dM[a, a] = -2.0 / ls[a] ** 2
            cols.append(np.concatenate([[0.0], _metric_columns(dM, ndim)]))
        return cols
    raise _cabi.TgpError("unsupported kernel for the B200 backend: %r" % (k,))


def lower_kernel_jacobian(kernel, ndim):
    """(``lower_kernel(kernel, ndim)``, J): J is the 4 x n_theta Jacobian of (ln amp, m00, m01, m11) with respect to
    ``kernel.theta`` -- columns in scikit-learn's theta order (a Product lists k1's then k2's), fixed
    hyper-parameters absent.  The chain rule that turns tgp_loglike_grad's derivatives into d logL / d theta
    (d logL / d theta = J^T g).  Accepts exactly what lower_kernel accepts."""
    desc = lower_kernel(kernel, ndim)

    def walk(k):
        if isinstance(k, Product):
            return walk(k.k1) + walk(k.k2)
        return _factor_jacobian(k, ndim)

    cols = walk(kernel)
    J = np.stack(cols, axis=1) if cols else np.zeros((4, 0))
    if J.shape[1] != len(kernel.theta):
        raise _cabi.TgpError("unsupported kernel for the B200 backend (theta layout): %r" % (kernel,))
    return desc, J


# ------------------------------------------------------------------------------------------------
# sums of stationary terms plus a white-noise level
# ------------------------------------------------------------------------------------------------
def _product_factors(k):
    """Factors of a (nested) Product in theta order."""
    if isinstance(k, Product):
        return _product_factors(k.k1) + _product_factors(k.k2)
    return [k]


def _expand_sum(k, ndim):
    """Distribute the constants of the tree k over its terms.  Returns (terms, whites, cols): terms is a list of
    TgpKernel (amp included), whites the list of white levels (scale included), and cols one entry per free
    hyper-parameter of k in theta order: (T, W) with T[c] = d (ln amp_c, m00_c, m01_c, m11_c) / d theta and
    W[j] = d white_j / d theta."""
    if isinstance(k, Sum):
        t1, w1, c1 = _expand_sum(k.k1, ndim)
        t2, w2, c2 = _expand_sum(k.k2, ndim)
        pad = [(np.vstack([T, np.zeros((len(t2), 4))]), np.concatenate([W, np.zeros(len(w2))])) for T, W in c1]
        pad += [(np.vstack([np.zeros((len(t1), 4)), T]), np.concatenate([np.zeros(len(w1)), W])) for T, W in c2]
        return t1 + t2, w1 + w2, pad
    if isinstance(k, WhiteKernel):
        lvl = float(k.noise_level)
        return [], [lvl], ([] if k.hyperparameter_noise_level.fixed else [(np.zeros((0, 4)), np.array([lvl]))])
    if isinstance(k, (Product, ConstantKernel)):
        factors = _product_factors(k)
        inner = [f for f in factors if not isinstance(f, ConstantKernel)]
        if len(inner) > 1:
            raise _cabi.TgpError("unsupported kernel for the B200 backend (more than one non-constant factor): %r"
                                 % (k,))
        if not inner:
            raise _cabi.TgpError("unsupported kernel for the B200 backend (a constant offset term): %r" % (k,))
        scale = float(np.prod([float(f.constant_value) for f in factors if isinstance(f, ConstantKernel)]))
        terms, whites, sub = _expand_sum(inner[0], ndim)
        for t in terms:
            t.amp *= scale
        whites = [scale * w for w in whites]
        cols = []
        for f in factors:
            if f is inner[0]:
                cols += [(T, scale * W) for T, W in sub]
            elif not f.hyperparameter_constant_value.fixed:   # d ln amp_c / d ln c = 1 for every term under it
                T = np.zeros((len(terms), 4))
                T[:, 0] = 1.0
                cols.append((T, np.array(whites)))
        return terms, whites, cols
    desc = lower_kernel(k, ndim)   # raises for anything that is not a supported stationary kernel
    return [desc], [], [(c[None, :], np.zeros(0)) for c in _factor_jacobian(k, ndim)]


def _lower_sum(kernel, ndim):
    terms, whites, cols = _expand_sum(kernel, ndim)
    if not terms:
        raise _cabi.TgpError("unsupported kernel for the B200 backend (no stationary term): %r" % (kernel,))
    if len(terms) > _cabi.MAX_TERMS:
        raise _cabi.TgpError("unsupported kernel for the B200 backend (%d stationary terms, at most %d): %r"
                             % (len(terms), _cabi.MAX_TERMS, kernel))
    desc = TgpKernelSum()
    desc.nterms, desc.ndim, desc.white = len(terms), ndim, float(sum(whites))
    for c, t in enumerate(terms):
        desc.term[c] = t
    return desc, whites, cols


def lower_kernel_sum(kernel, ndim):
    """sklearn kernel tree -> ``TgpKernelSum``.

    Accepted: Sum nodes; Products of any number of ``ConstantKernel`` factors and at most one other factor, which may
    itself be a Sum (the constants distribute over it); leaves are the stationary kernels ``lower_kernel`` accepts and
    ``WhiteKernel`` (possibly scaled; several add up).  Rejected with ``TgpError``: a product of two non-constant
    factors, a constant offset term, any other kernel, no stationary term, more than ``TGP_MAX_TERMS`` stationary
    terms.  Terms keep their order in the tree (k1 before k2)."""
    return _lower_sum(kernel, ndim)[0]


def lower_kernel_sum_jacobian(kernel, ndim):
    """(``lower_kernel_sum(kernel, ndim)``, J): J is the (4 nterms + 1) x n_theta Jacobian of (ln amp_c, m00_c, m01_c,
    m11_c for every term c, then ln white) with respect to ``kernel.theta`` -- columns in scikit-learn's theta order
    (Sum and Product list k1's then k2's), fixed hyper-parameters absent.  The ln white row is 0 when there is no
    white level.  d logL / d theta = J^T g with g from tgp_loglike_grad_sum."""
    desc, whites, cols = _lower_sum(kernel, ndim)
    n, w = desc.nterms, desc.white
    J = np.zeros((4 * n + 1, len(cols)))
    for j, (T, W) in enumerate(cols):
        J[: 4 * n, j] = T.reshape(-1)
        J[4 * n, j] = float(np.sum(W)) / w if w > 0 else 0.0
    if J.shape[1] != len(kernel.theta):
        raise _cabi.TgpError("unsupported kernel for the B200 backend (theta layout): %r" % (kernel,))
    return desc, J


def lower(kernel, ndim):
    """The device descriptor of a kernel: ``lower_kernel(kernel, ndim)`` whenever it accepts the kernel (every kernel
    that lowers to one term keeps that path), else ``lower_kernel_sum(kernel, ndim)``."""
    try:
        return lower_kernel(kernel, ndim)
    except _cabi.TgpError:
        return lower_kernel_sum(kernel, ndim)


def lower_jacobian(kernel, ndim):
    """``lower_kernel_jacobian`` or ``lower_kernel_sum_jacobian``, chosen as ``lower`` chooses."""
    try:
        return lower_kernel_jacobian(kernel, ndim)
    except _cabi.TgpError:
        return lower_kernel_sum_jacobian(kernel, ndim)


def descriptor_params(desc):
    """Every number of a descriptor (amplitudes, metrics, white level): a non-finite one cannot be factorised."""
    terms = [desc] if isinstance(desc, TgpKernel) else [desc.term[c] for c in range(desc.nterms)]
    vals = [v for t in terms for v in (t.amp, t.m00, t.m01, t.m11)]
    return vals if isinstance(desc, TgpKernel) else vals + [desc.white]
