"""GPU: the selected inverse (tgp_selinv), the analytic log-likelihood gradient (tgp_loglike_grad,
log_likelihood.log_likelihood_and_gradient, log_likelihood.ANALYTIC_GRADIENT) and the leave-one-out predictions
(GPInterpolation.loo_predict) -- against torch.cholesky_inverse, the numpy oracle, central differences of the device
log-likelihood, forward-difference fits and explicit refits."""
import numpy as np
import pytest
import torch

from oracle import gp_oracle as go
import grad_oracle as gro

pytestmark = pytest.mark.gpu

MI = np.array([[0.9, -0.35], [-0.35, 0.6]])
KSTR = {"rbf2": "2.0 * AnisotropicRBF(invLam=array([[0.9, -0.35], [-0.35, 0.6]]))",
        "vk2": "2.0 * AnisotropicVonKarman(invLam=array([[0.9, -0.35], [-0.35, 0.6]]))",
        "rbf1": "2.0 * RBF(0.8)",
        "m12": "1.5 * Matern(length_scale=0.12, nu=0.5)",
        "m32": "1.5 * Matern(length_scale=[0.3, 0.45], nu=1.5)",
        "m52": "ConstantKernel(1.5) * Matern(length_scale=0.4, nu=2.5)"}
FAMILY = {"rbf2": "rbf", "vk2": "vonkarman", "rbf1": "rbf", "m12": "matern12", "m32": "matern32", "m52": "matern52"}
# sizes of tests/test_gpu_envelope.py; the Matern supports (1e-40 of the amplitude) are 8-24 length scales long
SIZES = {"rbf2": (6000, 260.0), "vk2": (4500, 300.0), "rbf1": (5000, 900.0), "m12": (5000, 400.0),
         "m32": (5000, 400.0), "m52": (5000, 300.0)}


def _problem(case, n, field, seed=23):
    from treegp_b200 import backend, eval_kernel
    from treegp_b200.kernels import lower_kernel

    rng = np.random.default_rng(seed)
    ndim = 1 if case == "rbf1" else 2
    X = rng.uniform(0, field, size=(n, ndim))
    kern = eval_kernel(KSTR[case])
    desc = lower_kernel(kern, ndim)
    y = rng.normal(size=n)
    e2 = rng.uniform(0.005, 0.02, size=n)
    return X, y, e2, kern, desc


def _sorted_envelope(X, desc):
    """Points sorted along x and the envelope of K for that order (whether or not plan_envelope would take it)."""
    from treegp_b200 import backend

    Xd = backend.as_points(X)
    o = torch.argsort(Xd[:, 0], stable=True)
    dcut = backend.support_cutoffs(desc)[0]
    x = Xd[o, 0].cpu().numpy()
    return o, backend.envelope_rows(x, dcut)


def _inside(row_end, n):
    m = np.zeros((n, n), dtype=bool)
    for b, r in enumerate(row_end):
        m[512 * b:r, 512 * b:512 * (b + 1)] = True
    return m | m.T


@pytest.mark.parametrize("case", ["rbf2", "vk2", "rbf1", "m12", "m32", "m52"])
def test_selinv_dense_and_envelope_against_cholesky_inverse(gpu_ready, case):
    from treegp_b200 import backend

    n, field = SIZES[case]
    X, y, e2, kern, desc = _problem(case, n, field)
    o, re = _sorted_envelope(X, desc)
    Xs = backend.as_points(X)[o].contiguous()
    es = backend.to_device(e2)[o].contiguous()
    K = backend.kmat_sym(Xs, desc, es)[:, :n]
    ref = torch.cholesky_inverse(torch.linalg.cholesky(K)).cpu().numpy()
    A = backend.kmat_sym(Xs, desc, es, lower_only=True)
    B = A.clone()
    assert int(backend.potrf(A, n).item()) == 0 and int(backend.potrf(B, n, row_end=re).item()) == 0
    Zd = backend.selinv(A, n)[:, :n].cpu().numpy()
    Ze = backend.selinv(B, n, row_end=re)[:, :n].cpu().numpy()
    inside = _inside(re, n)
    scale = np.max(np.abs(ref))
    assert np.max(np.abs(Zd - ref)) <= 1e-9 * scale                      # dense: every entry, both triangles
    assert np.max(np.abs(Ze[inside] - ref[inside])) <= 1e-9 * scale
    assert np.max(np.abs(Ze[inside] - Zd[inside])) <= 1e-9 * scale
    if case in ("rbf2", "vk2", "rbf1"):
        assert not inside.all()
    # outside the envelope nothing was written: the K build's (tiny) entries and the never-touched upper triangle
    outside_lower = np.tril(~inside)
    assert np.array_equal(Ze[outside_lower], K.cpu().numpy()[outside_lower])


@pytest.mark.parametrize("case", ["rbf2", "vk2", "rbf1", "m12", "m32", "m52"])
def test_loglike_grad_against_the_oracle(gpu_ready, case):
    from treegp_b200 import backend

    n = 1500
    X, y, e2, kern, desc = _problem(case, n, 40.0 if case != "rbf1" else 300.0, seed=31)
    M = np.array([[desc.m00]]) if desc.ndim == 1 else np.array([[desc.m00, desc.m01], [desc.m01, desc.m11]])
    logl, g = gro.log_likelihood_gradient(FAMILY[case], X, y, e2, desc.amp, M)
    out, info, alpha, _ = backend.loglike_grad(backend.as_points(X), backend.to_device(y), backend.to_device(e2), desc)
    o = out.cpu().numpy()
    assert int(info.item()) == 0
    assert abs(o[0] - logl) <= 1e-9 * abs(logl)
    np.testing.assert_allclose(o[3:7], g, rtol=0, atol=1e-9 * np.max(np.abs(g)))
    _, ref_alpha = go.log_likelihood(go.kmat(FAMILY[case], X, amp=desc.amp, invLam=M) + np.diag(e2), y)
    np.testing.assert_allclose(alpha.cpu().numpy(), ref_alpha, rtol=0, atol=1e-9 * np.max(np.abs(ref_alpha)))


@pytest.mark.parametrize("case", ["rbf2", "vk2", "rbf1", "m12", "m32", "m52"])
@pytest.mark.parametrize("banded", [False, True])
def test_gradient_against_central_differences_of_the_device_loglike(gpu_ready, case, banded):
    import treegp_b200 as treegp

    n, field = 5000, (60.0 if case != "rbf1" else 900.0)
    X, y, e2, kern, desc = _problem(case, n, field, seed=41)
    ll = treegp.log_likelihood(X, y, np.sqrt(e2))
    ll.BANDED = banded
    v, g = ll.log_likelihood_and_gradient(kern)
    assert (getattr(ll, "n_banded_evaluations", 0) == 1) == banded
    assert ll.n_evaluations == 1
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

    n, field = SIZES["vk2"]
    X, y, e2, kern, desc = _problem("vk2", n, field)
    o, re = _sorted_envelope(X, desc)
    Xs, ys = backend.as_points(X)[o].contiguous(), backend.to_device(y)[o].contiguous()
    es = backend.to_device(e2)[o].contiguous()
    for row_end in (None, re):
        a = backend.loglike_grad(Xs, ys, es, desc, row_end=row_end)[0].cpu().numpy()
        b = backend.loglike_grad(Xs, ys, es, desc, row_end=row_end)[0].cpu().numpy()
        assert np.array_equal(a, b) and np.all(np.isfinite(a))
    e2b = e2.copy()
    e2b[3210] = -50.0
    eb = backend.to_device(e2b)[o].contiguous()
    for row_end in (None, re):
        out, info, _, _ = backend.loglike_grad(Xs, ys, eb, desc, row_end=row_end)
        out = out.cpu().numpy()
        assert int(info.item()) > 0 and out[0] == -np.inf and np.all(out[3:] == 0.0)
    assert _cabi.load().tgp_device_error(0) == 0


def test_fit_with_the_analytic_gradient(gpu_ready):
    """The problem of test_log_likelihood_search_with_and_without_the_envelope: same maximum with
    ANALYTIC_GRADIENT on and off, in fewer device evaluations."""
    import treegp_b200 as treegp
    from treegp_b200.log_likelihood import log_likelihood as LL
    from treegp_b200.two_pcf import get_correlation_length_matrix

    rng = np.random.default_rng(12)
    n, field = 4500, 70.0
    inv = np.linalg.inv(get_correlation_length_matrix(0.5, 0.2, 0.2))
    kstr = "4.0 * AnisotropicRBF(invLam=array([[%.17g, %.17g], [%.17g, %.17g]]))" % (inv[0, 0], inv[0, 1], inv[1, 0], inv[1, 1])
    X = rng.uniform(-field / 2, field / 2, size=(n, 2))
    kern = treegp.eval_kernel(kstr)
    y, y_err = treegp.sample_grf(kern, X, noise=0.05, seed=3)
    fits = {}
    saved = LL.ANALYTIC_GRADIENT
    try:
        for analytic in (False, True):
            LL.ANALYTIC_GRADIENT = analytic
            ll = treegp.log_likelihood(X, y, y_err)
            start = kern.clone_with_theta(kern.theta + np.array([0.2, -0.2, 0.1, 0.1]))
            k = ll.optimizer(start)
            fits[analytic] = (np.array(k.theta), ll._logL, ll.n_evaluations)
    finally:
        LL.ANALYTIC_GRADIENT = saved
    assert LL.ANALYTIC_GRADIENT is saved
    assert abs(fits[True][1] - fits[False][1]) <= 1e-7 * abs(fits[False][1])
    np.testing.assert_allclose(fits[True][0], fits[False][0], rtol=0, atol=5e-3)
    assert fits[True][2] < fits[False][2]


@pytest.mark.parametrize("banded", [False, True])
def test_loo_predict_against_explicit_refits(gpu_ready, monkeypatch, banded):
    """Dense: N = 400 in 2-D.  Envelope: 1-D points in a long field, with the envelope allowed at any N (at N = 1600
    it spans four block columns)."""
    import treegp_b200 as treegp
    from treegp_b200 import backend

    rng = np.random.default_rng(77)
    if banded:
        monkeypatch.setattr(backend, "ENVELOPE_MIN_N", 0)
        n, kstr = 1600, "2.0 * RBF(0.8)"
        X = rng.uniform(0, 200.0, size=(n, 1))
    else:
        n, kstr = 400, KSTR["vk2"]
        X = rng.uniform(0, 12.0, size=(n, 2))
    y = rng.normal(size=n) + 3.0
    yerr = rng.uniform(0.05, 0.15, size=n)
    gp = treegp.GPInterpolation(kernel=kstr, optimizer="none", normalize=True, white_noise=0.02)
    gp.initialize(X, y, y_err=yerr)
    mean_all = gp.predict(X[:5])      # a cached factor that loo_predict must leave alone
    factor = gp._factor[2].clone()
    mean, var = gp.loo_predict()
    assert torch.equal(factor, gp._factor[2])
    np.testing.assert_array_equal(gp.predict(X[:5]), mean_all)
    if banded:
        assert backend.plan_envelope(backend.as_points(X), gp._factor[1]) is not None
    resid = gp._y - gp._mean - gp._spatial_average
    for i in rng.choice(n, size=10, replace=False):
        keep = np.arange(n) != i
        g = treegp.GPInterpolation(kernel=kstr, optimizer="none", normalize=False)
        g.initialize(X[keep], resid[keep], y_err=gp._y_err[keep])
        m_i, c_i = g.return_gp_predict(resid[keep], X[keep], X[i:i + 1], g.kernel, y_err=gp._y_err[keep],
                                       return_cov=True)
        assert abs(mean[i] - (m_i[0] + gp._mean + gp._spatial_average[i])) <= 1e-8
        assert abs(var[i] - c_i[0, 0]) <= 1e-8
