"""GPU: sum kernels (several stationary terms plus a WhiteKernel level) -- the *_sum entry points against their
single-term twins (bit for bit for one term without white), against the numpy sum oracle (tests/sum_oracle.py) and
scikit-learn's GaussianProcessRegressor, central differences, repeatability, the -inf exit, the predictions of
GPInterpolation and the public log-likelihood fit."""
import numpy as np
import pytest
import torch

from oracle import gp_oracle as go
import sum_oracle as so

pytestmark = pytest.mark.gpu

VK2 = "AnisotropicVonKarman(invLam=array([[0.9, -0.35], [-0.35, 0.6]]))"
RBF2 = "AnisotropicRBF(invLam=array([[0.9, -0.35], [-0.35, 0.6]]))"
SINGLE = {"vk2": ("2.0 * " + VK2, 2), "rbf2": ("2.0 * " + RBF2, 2), "rbf1": ("2.0 * RBF(0.8)", 1),
          "m32": ("1.5 * Matern(length_scale=[0.3, 0.45], nu=1.5)", 2)}
SUMS = {"vk_rbf_white": ("2.0 * %s + 0.5 * RBF(3.0) + WhiteKernel(0.02)" % VK2, 2),
        "three_terms": ("1.5 * %s + ConstantKernel(0.7) * (Matern(0.5, nu=2.5) + 0.3 * %s) + WhiteKernel(0.01)"
                        % (VK2, RBF2), 2),
        "one_d": ("ConstantKernel(1.2) * VonKarman(0.9) + 0.4 * Matern(2.0, nu=0.5) + WhiteKernel(0.03)", 1)}


def _kernel(s):
    from treegp_b200 import eval_kernel

    return eval_kernel(s)


def _as_sum(desc):
    """A TgpKernel as a one-term TgpKernelSum with white = 0."""
    from treegp_b200 import _cabi

    d = _cabi.TgpKernelSum()
    d.nterms, d.ndim, d.white = 1, desc.ndim, 0.0
    d.term[0] = desc
    return d


def _sorted(X, desc, *arrays):
    """Points (and arrays) sorted along x, and the envelope of K for that order."""
    from treegp_b200 import backend

    Xd = backend.as_points(X)
    o = torch.argsort(Xd[:, 0], stable=True)
    x = Xd[o, 0].cpu().numpy()
    row_end = backend.envelope_rows(x, backend.support_cutoffs(desc)[0])
    return (Xd[o].contiguous(),) + tuple(backend.to_device(a)[o].contiguous() for a in arrays) + (row_end,)


def _eq(a, b):
    return torch.equal(a, b) if isinstance(a, torch.Tensor) else np.array_equal(a, b)


# ---- one term, no white: the single-term entries bit for bit -------------------------------------------------------
@pytest.mark.parametrize("case", list(SINGLE))
def test_one_term_sum_equals_the_single_term_entries(gpu_ready, case):
    from treegp_b200 import backend
    from treegp_b200.kernels import lower_kernel

    kstr, ndim = SINGLE[case]
    rng = np.random.default_rng(5)
    n, m, field = 5000, 20000, (300.0 if case == "vk2" else 250.0)
    X = rng.uniform(0, field, size=(n, ndim))
    X[100:110] = X[200:210]
    Xs = rng.uniform(0, field, size=(m, ndim))
    y = rng.normal(size=n)
    e2 = rng.uniform(0.005, 0.02, size=n)
    e2[100:110] += 3.0   # K stays positive definite with the von Karman rule between the coincident points
    e2[200:210] += 3.0
    d1 = lower_kernel(_kernel(kstr), ndim)
    ds = _as_sum(d1)
    e2d = backend.to_device(e2)
    assert _eq(backend.kmat_sym(X, d1, e2d), backend.kmat_sym(X, ds, e2d))
    assert _eq(torch.tril(backend.kmat_sym(X, d1, e2d, lower_only=True)[:, :n]),
               torch.tril(backend.kmat_sym(X, ds, e2d, lower_only=True)[:, :n]))
    assert _eq(backend.kmat_cross(Xs[:700], X, d1), backend.kmat_cross(Xs[:700], X, ds))
    Xo, yo, eo, row_end = _sorted(X, d1, y, e2)

    def zeroed():   # entries the calls do not write compare equal
        return torch.zeros((n + 1, backend.even(n)), dtype=torch.float64, device=Xo.device)

    for re in (None, row_end):
        for want_alpha in (False, True):
            a = backend.loglike(Xo, yo, eo, d1, work=zeroed(), want_alpha=want_alpha, row_end=re)
            b = backend.loglike(Xo, yo, eo, ds, work=zeroed(), want_alpha=want_alpha, row_end=re)
            assert all(_eq(u, v) for u, v in zip(a, b))
        g1, _, alpha, L1 = backend.loglike_grad(Xo, yo, eo, d1, work=zeroed(), row_end=re)
        gs, _, _, Ls = backend.loglike_grad(Xo, yo, eo, ds, work=zeroed(), row_end=re)
        assert _eq(g1, gs[:7]) and gs[7].item() == 0.0 and _eq(L1, Ls)
        for trunc in (False, True):
            assert _eq(backend.predict_mean(Xs, Xo, d1, alpha, truncate=trunc),
                       backend.predict_mean(Xs, Xo, ds, alpha, truncate=trunc))
        L = backend.loglike(Xo, yo, eo, d1, want_alpha=True, row_end=re)[3]
        assert _eq(backend.predict_var(Xs[:3000], Xo, d1, L, row_end=re),
                   backend.predict_var(Xs[:3000], Xo, ds, L, row_end=re))
    s1, ss = {}, {}
    v1 = backend.predict_var_windowed(Xs, Xo, d1, eo, stats=s1)
    vs = backend.predict_var_windowed(Xs, Xo, ds, eo, stats=ss)
    assert s1 == ss
    if v1 is not None:
        assert _eq(v1, vs)


# ---- values against the oracle --------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", list(SUMS))
def test_sum_kmat_against_the_oracle(gpu_ready, case):
    """Duplicated points: a von Karman term is 0 between distinct coincident points, the other terms are not, and the
    white level sits on the diagonal only (never in K(Xs, X), even for Xs = X)."""
    from treegp_b200 import backend
    from treegp_b200.kernels import lower_kernel_sum

    kstr, ndim = SUMS[case]
    rng = np.random.default_rng(8)
    X = rng.uniform(0, 8.0, size=(700, ndim))
    X[50:60] = X[300:310]
    Xs = rng.uniform(0, 8.0, size=(300, ndim))
    d = lower_kernel_sum(_kernel(kstr), ndim)
    terms, white = so.terms_of(d)
    amp = sum(t[1] for t in terms)
    diag = rng.uniform(0.01, 0.02, size=700)
    K = backend.kmat_sym(X, d, backend.to_device(diag))[:, :700].cpu().numpy()
    np.testing.assert_allclose(K, so.sum_kmat(terms, X, white=white) + np.diag(diag), rtol=0, atol=2e-13 * amp)
    Kx = backend.kmat_cross(Xs, X, d)[:, :700].cpu().numpy()
    np.testing.assert_allclose(Kx, so.sum_kmat(terms, Xs, X), rtol=0, atol=2e-13 * amp)
    Kxx = backend.kmat_cross(X, X, d)[:, :700].cpu().numpy()
    np.testing.assert_allclose(np.diag(Kxx), amp, rtol=1e-15)
    # the quirk is per term: the sum between coincident points is the non-von-Karman amplitude
    vk_amp = sum(t[1] for t in terms if t[0] == "vonkarman")
    assert K[50, 300] == pytest.approx(amp - vk_amp, rel=1e-14)
    # the sklearn kernel itself evaluates the same matrix (the device evaluates every term of the sklearn tree)
    np.testing.assert_allclose(_kernel(kstr)(X), so.sum_kmat(terms, X, white=white), rtol=0, atol=2e-13 * amp)


@pytest.mark.parametrize("case", list(SUMS))
@pytest.mark.parametrize("banded", [False, True])
def test_loglike_and_gradient_against_the_oracle(gpu_ready, case, banded):
    from treegp_b200 import backend
    from treegp_b200.kernels import lower_kernel_sum

    kstr, ndim = SUMS[case]
    rng = np.random.default_rng(31)
    n = 2500
    X = rng.uniform(0, 120.0 if ndim == 2 else 600.0, size=(n, ndim))
    y = rng.normal(size=n)
    e2 = rng.uniform(0.005, 0.02, size=n)
    d = lower_kernel_sum(_kernel(kstr), ndim)
    Xo, yo, eo, row_end = _sorted(X, d, y, e2)
    if banded:
        assert row_end[0] < n     # a real envelope
    out = backend.loglike_grad(Xo, yo, eo, d, row_end=row_end if banded else None)[0].cpu().numpy()
    ll = backend.loglike(Xo, yo, eo, d, row_end=row_end if banded else None)[0].cpu().numpy()
    terms, white = so.terms_of(d)
    ref, g = so.sum_log_likelihood_gradient(terms, white, Xo.cpu().numpy(), yo.cpu().numpy(), eo.cpu().numpy())
    assert out.shape == (4 + 4 * d.nterms,)
    assert out[0] == pytest.approx(ref, rel=1e-10) and ll[0] == pytest.approx(ref, rel=1e-10)
    np.testing.assert_allclose(out[3:], g, rtol=0, atol=1e-6 * np.max(np.abs(g)))


def test_loglike_and_gradient_against_sklearn(gpu_ready):
    """scikit-learn's GaussianProcessRegressor(kernel, alpha=y_err**2).log_marginal_likelihood(theta,
    eval_gradient=True): the reference's formula and its theta gradient, through the public class."""
    import treegp_b200 as treegp
    from sklearn.gaussian_process import GaussianProcessRegressor

    kstr = ("ConstantKernel(2.0) * RBF([0.7, 1.3]) + ConstantKernel(0.5) * Matern(1.1, nu=1.5) "
            "+ WhiteKernel(0.05) + ConstantKernel(0.3) * Matern(0.4, nu=0.5)")
    rng = np.random.default_rng(4)
    n = 1500
    X = rng.uniform(0, 25.0, size=(n, 2))
    y = rng.normal(size=n)
    yerr = rng.uniform(0.05, 0.15, size=n)
    k = _kernel(kstr)
    ref, ref_g = GaussianProcessRegressor(kernel=k, alpha=yerr ** 2, optimizer=None).fit(X, y).log_marginal_likelihood(
        k.theta, eval_gradient=True)
    ll = treegp.log_likelihood(X, y, yerr)
    v, g = ll.log_likelihood_and_gradient(k)
    assert v == pytest.approx(ref, rel=1e-10)
    assert ll.log_likelihood(k) == pytest.approx(ref, rel=1e-10)
    np.testing.assert_allclose(g, ref_g, rtol=0, atol=1e-6 * np.max(np.abs(ref_g)))


@pytest.mark.parametrize("case", list(SUMS))
@pytest.mark.parametrize("banded", [False, True])
def test_gradient_against_central_differences_of_the_device_loglike(gpu_ready, case, banded):
    import treegp_b200 as treegp

    kstr, ndim = SUMS[case]
    rng = np.random.default_rng(41)
    n = 5000
    X = rng.uniform(0, 300.0 if ndim == 2 else 900.0, size=(n, ndim))
    y = rng.normal(size=n)
    e2 = rng.uniform(0.005, 0.02, size=n)
    kern = _kernel(kstr)
    ll = treegp.log_likelihood(X, y, np.sqrt(e2))
    ll.BANDED = banded
    v, g = ll.log_likelihood_and_gradient(kern)
    assert (getattr(ll, "n_banded_evaluations", 0) == 1) == banded
    assert v == pytest.approx(ll.log_likelihood(kern), rel=1e-11)
    theta = np.array(kern.theta)
    h = 1e-5
    fd = np.empty_like(theta)
    for j in range(len(theta)):
        e = np.zeros_like(theta)
        e[j] = h
        fd[j] = (ll.log_likelihood(kern.clone_with_theta(theta + e))
                 - ll.log_likelihood(kern.clone_with_theta(theta - e))) / (2 * h)
    np.testing.assert_allclose(g, fd, rtol=0, atol=1e-5 * np.max(np.abs(fd)))


def test_repeated_calls_are_bit_identical_and_failures_give_minus_inf(gpu_ready):
    from treegp_b200 import _cabi, backend
    from treegp_b200.kernels import lower_kernel_sum

    kstr, ndim = SUMS["three_terms"]
    rng = np.random.default_rng(2)
    n = 4500
    X = rng.uniform(0, 300.0, size=(n, ndim))
    y = rng.normal(size=n)
    e2 = rng.uniform(0.005, 0.02, size=n)
    d = lower_kernel_sum(_kernel(kstr), ndim)
    Xo, yo, eo, row_end = _sorted(X, d, y, e2)
    for re in (None, row_end):
        a = backend.loglike_grad(Xo, yo, eo, d, row_end=re)[0].cpu().numpy()
        b = backend.loglike_grad(Xo, yo, eo, d, row_end=re)[0].cpu().numpy()
        assert np.array_equal(a, b) and np.all(np.isfinite(a))
    e2b = e2.copy()
    e2b[3210] = -50.0
    eb = backend.to_device(e2b)[torch.argsort(backend.as_points(X)[:, 0], stable=True)].contiguous()
    for re in (None, row_end):
        out, info, _, _ = backend.loglike_grad(Xo, yo, eb, d, row_end=re)
        out = out.cpu().numpy()
        assert int(info.item()) > 0 and out[0] == -np.inf and np.all(out[3:] == 0.0)
    assert _cabi.load().tgp_device_error(0) == 0


# ---- predictions through GPInterpolation ---------------------------------------------------------------------------
@pytest.mark.parametrize("banded", [False, True])
def test_predictions_with_a_sum_kernel(gpu_ready, monkeypatch, banded):
    """Dense: N = 900 in 2-D.  Envelope: 1-D points in a long field, with the envelope allowed at any N."""
    import treegp_b200 as treegp
    from treegp_b200 import backend
    from treegp_b200.kernels import lower_kernel_sum

    rng = np.random.default_rng(17)
    if banded:
        monkeypatch.setattr(backend, "ENVELOPE_MIN_N", 0)
        n, field, ndim, kstr = 1600, 200.0, 1, "2.0 * RBF(0.8) + 0.5 * VonKarman(1.5) + WhiteKernel(0.02)"
    else:
        n, field, ndim, kstr = 900, 12.0, 2, SUMS["vk_rbf_white"][0]
    X = rng.uniform(0, field, size=(n, ndim))
    Xs = rng.uniform(0, field, size=(400, ndim))
    y = rng.normal(size=n)
    yerr = rng.uniform(0.05, 0.15, size=n)
    gp = treegp.GPInterpolation(kernel=kstr, optimizer="none", normalize=False)
    gp.initialize(X, y, y_err=yerr)
    gp.solve()
    mean, cov = gp.predict(Xs, return_cov=True)
    assert (gp._envelope is not None) == banded
    terms, white = so.terms_of(lower_kernel_sum(_kernel(kstr), ndim))
    K = so.sum_kmat(terms, X, white=white) + np.diag(yerr ** 2)
    _, rmean, rcov = go.gp_predict(K, so.sum_kmat(terms, Xs, X), so.sum_kmat(terms, Xs, white=white), y)
    scale = np.max(np.abs(rmean))
    np.testing.assert_allclose(mean, rmean, rtol=0, atol=1e-9 * scale)
    np.testing.assert_allclose(cov, rcov, rtol=0, atol=1e-9)
    assert np.all(np.diag(cov) > white)        # white on the diagonal of kernel(X2)
    for windowed in (False, True):
        gp.WINDOWED_VARIANCE = windowed
        m2, var = gp.predict_var(Xs)
        np.testing.assert_allclose(m2, rmean, rtol=0, atol=1e-9 * scale)
        np.testing.assert_allclose(var, np.diag(rcov), rtol=0, atol=1e-9)
    assert gp.return_log_likelihood() == pytest.approx(go.log_likelihood(K, y)[0], rel=1e-10)
    # leave-one-out against explicit refits
    lmean, lvar = gp.loo_predict()
    for i in rng.choice(n, size=8, replace=False):
        keep = np.arange(n) != i
        g = treegp.GPInterpolation(kernel=kstr, optimizer="none", normalize=False)
        g.initialize(X[keep], y[keep], y_err=yerr[keep])
        m_i, c_i = g.return_gp_predict(y[keep], X[keep], X[i:i + 1], g.kernel, y_err=yerr[keep], return_cov=True)
        assert abs(lmean[i] - m_i[0]) <= 1e-8
        assert abs(lvar[i] - c_i[0, 0]) <= 1e-8


# ---- the public fit ------------------------------------------------------------------------------------------------
def test_fit_of_a_noise_level(gpu_ready):
    """A von Karman field plus white noise of a known level: the log-likelihood fit finds the same maximum with
    forward differences and with the analytic gradient, and that maximum is the one of a scipy L-BFGS-B fit of the
    numpy oracle."""
    import treegp_b200 as treegp
    from scipy import optimize
    from treegp_b200.kernels import lower_kernel_sum_jacobian
    from treegp_b200.log_likelihood import log_likelihood as LL

    rng = np.random.default_rng(21)
    n, field, w_true = 500, 12.0, 0.04
    X = rng.uniform(0, field, size=(n, 2))
    # the field: a draw of 1.5 * von Karman (numpy, from the oracle's K), measurement errors 0.02, white level w_true
    K = go.kmat("vonkarman", X, amp=1.5, invLam=np.array([[0.8, 0.15], [0.15, 0.5]]))
    y = np.linalg.cholesky(K + 1e-10 * np.eye(n)) @ rng.normal(size=n)
    yerr = np.full(n, 0.02)
    y = y + rng.normal(scale=0.02, size=n) + rng.normal(scale=np.sqrt(w_true), size=n)
    start = "1.0 * AnisotropicVonKarman(invLam=array([[0.7, 0.15], [0.15, 0.5]])) + WhiteKernel(0.01)"
    fits = {}
    saved = LL.ANALYTIC_GRADIENT
    try:
        for analytic in (False, True):
            LL.ANALYTIC_GRADIENT = analytic
            gp = treegp.GPInterpolation(kernel=start, optimizer="log-likelihood", normalize=False)
            gp.initialize(X, y, y_err=yerr)
            gp.solve()
            fits[analytic] = (np.array(gp.kernel.theta), gp._optimizer._logL, gp._optimizer.n_evaluations)
    finally:
        LL.ANALYTIC_GRADIENT = saved
    np.testing.assert_allclose(fits[True][0], fits[False][0], rtol=0, atol=5e-3)
    assert fits[True][2] < fits[False][2]
    k0 = _kernel(start)

    def minus(theta):
        desc, J = lower_kernel_sum_jacobian(k0.clone_with_theta(theta), 2)
        terms, white = so.terms_of(desc)
        v, g = so.sum_log_likelihood_gradient(terms, white, X, y, yerr ** 2)
        return -v, -(J.T @ g)

    ref = optimize.minimize(minus, k0.theta, method="L-BFGS-B", jac=True)
    for analytic in (False, True):
        assert fits[analytic][1] == pytest.approx(-ref.fun, rel=1e-6)
    w_fit = np.exp(fits[True][0][-1])
    assert 0.5 * w_true < w_fit < 2.0 * w_true
