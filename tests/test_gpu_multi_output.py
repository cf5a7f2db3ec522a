"""GPU: several outputs sharing one kernel -- the multi-output entries against r single-output runs (bit for bit per
column), against the numpy joint oracle (tests/multi_oracle.py) and central differences, repeatability and the -inf
exit, and the public API (GPInterpolation, log_likelihood) against single-output instances and a scipy fit."""
import numpy as np
import pytest
import torch

import multi_oracle as mo
import sum_oracle as so

pytestmark = pytest.mark.gpu

VK2 = "AnisotropicVonKarman(invLam=array([[0.9, -0.35], [-0.35, 0.6]]))"
CASES = {"single": "2.0 * " + VK2, "sum_white": "2.0 * %s + 0.5 * RBF(3.0) + WhiteKernel(0.02)" % VK2}
# 1-D coordinates: kernel string and field length (long enough for an envelope at N = 5000)
CASES_1D = {"single_1d": ("2.0 * VonKarman(0.9)", 1000.0),
            "sum_1d": ("ConstantKernel(1.2) * VonKarman(0.9) + 0.4 * Matern(2.0, nu=0.5) + WhiteKernel(0.03)", 1000.0)}


def _kernel(s):
    from treegp_b200 import eval_kernel

    return eval_kernel(s)


def _desc(kstr, ndim=2):
    from treegp_b200.kernels import lower

    return lower(_kernel(kstr), ndim)


def _field(n, r, field, seed, ndim=2):
    rng = np.random.default_rng(seed)
    X = rng.uniform(0, field, size=(n, ndim))
    Y = rng.normal(size=(n, r))
    e2 = rng.uniform(0.005, 0.02, size=n)
    return X, Y, e2


def _sorted(X, desc, Y, e2):
    """Points, outputs and errors sorted along x, and the envelope of K for that order."""
    from treegp_b200 import backend

    Xd = backend.as_points(X)
    o = torch.argsort(Xd[:, 0], stable=True)
    row_end = backend.envelope_rows(Xd[o, 0].cpu().numpy(), backend.support_cutoffs(desc)[0])
    return Xd[o].contiguous(), backend.to_device(Y)[o].contiguous(), backend.to_device(e2)[o].contiguous(), row_end


@pytest.mark.parametrize("r", [1, 2, 3, 8])
@pytest.mark.parametrize("case", list(CASES) + list(CASES_1D))
def test_outputs_as_columns_against_single_output_runs(gpu_ready, case, r):
    """Each column of alpha (K^-1 Y and L^-1 Y) and of the truncated mean is its single-output run bit for bit; the
    joint logL and gradient are the sums of the single-output ones; with r = 1 everything is bit for bit."""
    from treegp_b200 import backend

    kstr, field, ndim = (CASES[case], 300.0, 2) if case in CASES else CASES_1D[case] + (1,)
    d = _desc(kstr, ndim)
    X, Y, e2 = _field(5000, r, field, 5 + r, ndim)
    Xo, Yo, eo, row_end = _sorted(X, d, Y, e2)
    assert row_end[0] < 5000      # a real envelope
    Xs = backend.as_points(np.random.default_rng(9).uniform(0, field, size=(20000, ndim)))
    for re in (None, row_end):
        for want_alpha in (False, True):
            out, info, alpha, _ = backend.loglike(Xo, Yo, eo, d, want_alpha=want_alpha, row_end=re)
            singles = [backend.loglike(Xo, Yo[:, c].contiguous(), eo, d, want_alpha=want_alpha, row_end=re)
                       for c in range(r)]
            assert int(info.item()) == 0
            for c in range(r):
                assert torch.equal(alpha[:, c], singles[c][2]), (re is None, want_alpha, c)
            ll = [float(s[0][0].item()) for s in singles]
            if r == 1:
                assert torch.equal(out, singles[0][0])
            assert float(out[0].item()) == pytest.approx(sum(ll), rel=1e-12)
            assert float(out[2].item()) == float(singles[0][0][2].item())    # logdet once, as the single output
        g, _, galpha, _ = backend.loglike_grad(Xo, Yo, eo, d, row_end=re)
        gs = [backend.loglike_grad(Xo, Yo[:, c].contiguous(), eo, d, row_end=re)[0] for c in range(r)]
        k = len(gs[0])
        if r == 1:
            assert torch.equal(g[:k], gs[0])
        assert torch.equal(galpha, alpha)
        tot = torch.stack(gs).sum(dim=0)
        tot[2] = gs[0][2]                       # the joint record carries logdet once
        torch.testing.assert_close(g[:k], tot, rtol=1e-10, atol=1e-10 * float(tot[3:].abs().max()))
        mt = backend.predict_mean(Xs, Xo, d, alpha, truncate=True)
        mf = backend.predict_mean(Xs, Xo, d, alpha, truncate=False)
        for c in range(r):
            st = backend.predict_mean(Xs, Xo, d, alpha[:, c].contiguous(), truncate=True)
            assert torch.equal(mt[:, c], st), c
            # the full sum splits the training points over CTAs (M alone does not fill the machine) and adds the
            # partial sums with atomics in whatever order they arrive, for one output as for several: two calls differ
            # where the partials cancel, measured up to 4e-14 of the largest mean value (1-D, 8 partials per point)
            sf = backend.predict_mean(Xs, Xo, d, alpha[:, c].contiguous(), truncate=False)
            torch.testing.assert_close(mf[:, c], sf, rtol=1e-14, atol=2e-13 * float(sf.abs().max()))
        torch.testing.assert_close(mt, mf, rtol=1e-14, atol=2e-13 * float(mf.abs().max()))


@pytest.mark.parametrize("n", [5000, 20000])
def test_multi_column_sweeps_equal_single_column_sweeps(gpu_ready, n):
    """tgp_potrs_multi streams the factor once for r columns (groups of 2, 4 or 8, padded with zero columns); every
    column equals its own tgp_potrs_vec solve bit for bit, and repeats are bit-identical.  N = 20000 gives several
    slabs per CTA."""
    from treegp_b200 import backend

    d = _desc(CASES["single"])
    X, Y, e2 = _field(n, 8, 300.0 * np.sqrt(n / 5000.0), 29)
    Xo, Yo, eo, row_end = _sorted(X, d, Y, e2)
    _, info, _, ws = backend.loglike(Xo, Yo[:, 0].contiguous(), eo, d, row_end=row_end)
    assert int(info.item()) == 0
    ld = ws.stride(0)
    singles = []
    for c in range(8):
        b = Yo[:, c].contiguous()
        singles.append(backend.potrs_vec(ws, n, b))
    for r in range(1, 9):
        B = torch.zeros((r, ld), dtype=torch.float64, device=Xo.device)
        B[:, :n] = Yo[:, :r].T
        B2 = B.clone()
        backend.potrs_multi(ws, n, B)
        backend.potrs_multi(ws, n, B2)
        assert torch.equal(B, B2)
        for c in range(r):
            assert torch.equal(B[c, :n], singles[c]), (r, c)


def test_full_mean_of_columns_equals_single_output_bit_for_bit(gpu_ready):
    """With enough test points to fill the machine there is no split: each column of the full multi-output mean is its
    single-output mean bit for bit."""
    from treegp_b200 import backend

    for kstr in CASES.values():
        d = _desc(kstr)
        X, Y, _ = _field(700, 3, 300.0, 2)
        Xd = backend.as_points(X)
        alpha = backend.to_device(Y)
        Xs = backend.as_points(np.random.default_rng(3).uniform(0, 300.0, size=(1 << 18, 2)))
        m = backend.predict_mean(Xs, Xd, d, alpha, truncate=False)
        for c in range(3):
            assert torch.equal(m[:, c], backend.predict_mean(Xs, Xd, d, alpha[:, c].contiguous(), truncate=False))


@pytest.mark.parametrize("banded", [False, True])
@pytest.mark.parametrize("case", list(CASES))
def test_joint_loglike_and_gradient_of_columns_against_the_oracle(gpu_ready, monkeypatch, case, banded):
    from treegp_b200 import backend
    from treegp_b200.kernels import lower_jacobian
    from treegp_b200.log_likelihood import log_likelihood as LL

    k = _kernel(CASES[case])
    d = _desc(CASES[case])
    X, Y, e2 = _field(700, 3, 200.0, 11)
    Xo, Yo, eo, row_end = _sorted(X, d, Y, e2)
    if banded:
        assert row_end[0] < 700
    out = backend.loglike_grad(Xo, Yo, eo, d, row_end=row_end if banded else None)[0].cpu().numpy()
    terms, white = so.terms_of(backend.as_sum(d))
    ll, g, _ = mo.joint_log_likelihood_gradient(terms, white, X, Y, e2)
    assert out[0] == pytest.approx(ll, rel=1e-10)
    np.testing.assert_allclose(out[3:], g, rtol=1e-7, atol=1e-9 * np.max(np.abs(g)))
    # the public class, in sklearn's theta, against central differences of its own joint logL
    if banded:
        monkeypatch.setattr(backend, "ENVELOPE_MIN_N", 0)
    lik = LL(X, Y, np.sqrt(e2))
    v, gt = lik.log_likelihood_and_gradient(k)
    assert v == pytest.approx(ll, rel=1e-10)
    _, J = lower_jacobian(k, 2)
    np.testing.assert_allclose(gt, J.T @ g[:J.shape[0]], rtol=1e-7, atol=1e-9 * np.max(np.abs(gt)))
    h = 1e-5
    fd = []
    for i in range(len(k.theta)):
        tp, tm = k.theta.copy(), k.theta.copy()
        tp[i] += h
        tm[i] -= h
        fd.append((lik.log_likelihood(k.clone_with_theta(tp)) - lik.log_likelihood(k.clone_with_theta(tm))) / (2 * h))
    np.testing.assert_allclose(gt, fd, rtol=2e-5, atol=1e-6 * np.max(np.abs(gt)))


def test_repeated_calls_with_columns_are_bit_identical_and_failures_give_minus_inf(gpu_ready):
    from treegp_b200 import backend

    d = _desc(CASES["sum_white"])
    X, Y, e2 = _field(5000, 4, 300.0, 13)
    Xo, Yo, eo, row_end = _sorted(X, d, Y, e2)
    Xs = backend.as_points(np.random.default_rng(1).uniform(0, 300.0, size=(30000, 2)))
    for re in (None, row_end):
        a = backend.loglike_grad(Xo, Yo, eo, d, row_end=re)
        b = backend.loglike_grad(Xo, Yo, eo, d, row_end=re)
        assert torch.equal(a[0], b[0]) and torch.equal(a[2], b[2])
        assert torch.equal(backend.predict_mean(Xs, Xo, d, a[2], truncate=True),
                           backend.predict_mean(Xs, Xo, d, a[2], truncate=True))
        bad = eo.clone()
        bad[100] = -1e3                         # not positive definite
        out, info, _, _ = backend.loglike_grad(Xo, Yo, bad, d, row_end=re)
        o = out.cpu().numpy()
        assert int(info.item()) > 0 and o[0] == -np.inf and np.all(o[3:] == 0.0)
        assert float(backend.loglike(Xo, Yo, bad, d, row_end=re)[0][0].item()) == -np.inf


@pytest.mark.parametrize("banded", [False, True])
def test_gp_interpolation_with_several_outputs(gpu_ready, monkeypatch, banded):
    """predict, return_cov, predict_var, loo_predict and return_log_likelihood of a 3-output GPInterpolation against
    three single-output ones with the same kernel."""
    import treegp_b200 as treegp
    from treegp_b200 import backend

    if banded:
        monkeypatch.setattr(backend, "ENVELOPE_MIN_N", 0)
    kstr = CASES["sum_white"]
    X, Y, e2 = _field(1500, 3, 150.0, 17)
    Y = Y + np.array([1.0, -2.0, 0.5])
    Xs = np.random.default_rng(2).uniform(0, 150.0, size=(400, 2))
    gp = treegp.GPInterpolation(kernel=kstr, optimizer="none", normalize=True, white_noise=0.01)
    gp.initialize(X, Y, y_err=np.sqrt(e2))
    gp.solve()
    mean, cov = gp.predict(Xs, return_cov=True)
    pm, pv = gp.predict_var(Xs)
    lm, lv = gp.loo_predict()
    assert mean.shape == (400, 3) and cov.shape == (400, 400) and pm.shape == (400, 3) and pv.shape == (400,)
    assert lm.shape == (1500, 3) and lv.shape == (1500,) and gp._alpha.shape == (1500, 3) and gp._mean.shape == (3,)
    lls = 0.0
    for c in range(3):
        g1 = treegp.GPInterpolation(kernel=kstr, optimizer="none", normalize=True, white_noise=0.01)
        g1.initialize(X, Y[:, c], y_err=np.sqrt(e2))
        g1.solve()
        m1, c1 = g1.predict(Xs, return_cov=True)
        np.testing.assert_allclose(mean[:, c], m1, rtol=1e-11, atol=1e-11)
        np.testing.assert_array_equal(gp._alpha[:, c], g1._alpha)
        np.testing.assert_allclose(cov, c1, rtol=1e-12, atol=1e-13)
        v1 = g1.predict_var(Xs)
        np.testing.assert_allclose(pm[:, c], v1[0], rtol=1e-11, atol=1e-11)
        np.testing.assert_allclose(pv, v1[1], rtol=1e-12, atol=1e-13)
        l1 = g1.loo_predict()
        np.testing.assert_allclose(lm[:, c], l1[0], rtol=1e-11, atol=1e-11)
        np.testing.assert_allclose(lv, l1[1], rtol=1e-12, atol=1e-13)
        lls += g1.return_log_likelihood()
    assert gp.return_log_likelihood() == pytest.approx(lls, rel=1e-12)


def test_fit_of_a_shared_kernel(gpu_ready):
    """Two outputs drawn from one RBF GP: the public "log-likelihood" fit reaches the maximum of a scipy L-BFGS-B fit
    of the numpy joint oracle -- to 1e-5 in theta with the analytic gradient; with forward differences (gradient
    noise ~ 1e-8 |logL| / step) to the same logL and 1e-3 in theta."""
    import treegp_b200 as treegp
    from scipy import optimize
    from treegp_b200.kernels import lower_kernel_sum_jacobian
    from treegp_b200.log_likelihood import log_likelihood as LL
    from oracle import gp_oracle as go

    rng = np.random.default_rng(23)
    n = 400
    X = rng.uniform(0, 10.0, size=(n, 2))
    K = go.kmat("rbf", X, amp=1.5, invLam=np.array([[0.8, 0.15], [0.15, 0.5]]))
    Lk = np.linalg.cholesky(K + 1e-8 * np.eye(n))
    Y = np.stack([Lk @ rng.normal(size=n) for _ in range(2)], axis=1) + rng.normal(scale=0.05, size=(n, 2))
    yerr = np.full(n, 0.05)
    start = "1.0 * AnisotropicRBF(invLam=array([[0.6, 0.1], [0.1, 0.6]]))"
    k0 = _kernel(start)

    def minus(theta):
        desc, J = lower_kernel_sum_jacobian(k0.clone_with_theta(theta), 2)
        terms, white = so.terms_of(desc)
        v, g, _ = mo.joint_log_likelihood_gradient(terms, white, X, Y, yerr ** 2)
        return -v, -(J.T @ g)

    ref = optimize.minimize(minus, k0.theta, method="L-BFGS-B", jac=True)
    saved = LL.ANALYTIC_GRADIENT
    try:
        for analytic in (True, False):
            LL.ANALYTIC_GRADIENT = analytic
            gp = treegp.GPInterpolation(kernel=start, optimizer="log-likelihood", normalize=False)
            gp.initialize(X, Y, y_err=yerr)
            gp.solve()
            theta = np.array(gp.kernel.theta)
            np.testing.assert_allclose(theta, ref.x, rtol=0, atol=1e-5 if analytic else 1e-3)
            assert gp._optimizer._logL == pytest.approx(-ref.fun, rel=1e-7)
    finally:
        LL.ANALYTIC_GRADIENT = saved
