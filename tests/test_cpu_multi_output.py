"""CPU: several outputs sharing one kernel without a GPU -- the numpy joint-likelihood oracle against scikit-learn's
GaussianProcessRegressor on multi-target y and against the single-output oracles, the host-side validation of a 2-D y
in GPInterpolation, and argument validation of the multi-output C entry points."""
import ctypes

import numpy as np
import pytest

import multi_oracle as mo
import sum_oracle as so

SKLEARN_KERNELS = [
    ("ConstantKernel(2.0) * RBF([0.6, 1.1])", 2, 3),
    ("ConstantKernel(0.8) * Matern(0.5, nu=1.5) + ConstantKernel(0.5) * RBF(2.0) + WhiteKernel(0.05)", 1, 2),
    ("ConstantKernel(1.5) * Matern(0.7, nu=2.5) + WhiteKernel(0.02)", 2, 8),
]


def _kernel(s):
    from treegp_b200 import eval_kernel

    return eval_kernel(s)


def _data(ndim, r, n=120, seed=0):
    rng = np.random.default_rng(seed + 10 * ndim + r)
    X = rng.uniform(0, 5, size=(n, ndim))
    X[7] = X[3]                                  # a duplicated point
    return X, rng.normal(size=(n, r)), rng.uniform(0.01, 0.03, size=n)


@pytest.mark.parametrize("kstr,ndim,r", SKLEARN_KERNELS)
def test_joint_oracle_against_sklearn_multi_target(kstr, ndim, r):
    """GaussianProcessRegressor(kernel, alpha=y_err**2).log_marginal_likelihood(theta, eval_gradient=True) with y of
    shape (n, r) sums the per-target values and gradients: the oracle's joint value and gradient."""
    from sklearn.gaussian_process import GaussianProcessRegressor
    from treegp_b200.kernels import lower_kernel_sum_jacobian

    X, Y, e2 = _data(ndim, r)
    k = _kernel(kstr)
    gpr = GaussianProcessRegressor(kernel=k, alpha=e2, optimizer=None).fit(X, Y)
    ref, ref_g = gpr.log_marginal_likelihood(k.theta, eval_gradient=True)
    desc, J = lower_kernel_sum_jacobian(k, ndim)
    terms, white = so.terms_of(desc)
    logl, g, _ = mo.joint_log_likelihood_gradient(terms, white, X, Y, e2)
    assert logl == pytest.approx(ref, rel=1e-10)
    np.testing.assert_allclose(J.T @ g, ref_g, rtol=1e-7, atol=1e-8 * np.max(np.abs(ref_g)))


@pytest.mark.parametrize("kstr,ndim,r", SKLEARN_KERNELS)
def test_joint_gradient_is_the_sum_of_single_output_gradients(kstr, ndim, r):
    from treegp_b200.kernels import lower_kernel_sum

    X, Y, e2 = _data(ndim, r, seed=1)
    terms, white = so.terms_of(lower_kernel_sum(_kernel(kstr), ndim))
    logl, g, A = mo.joint_log_likelihood_gradient(terms, white, X, Y, e2)
    singles = [so.sum_log_likelihood_gradient(terms, white, X, Y[:, c], e2) for c in range(r)]
    assert logl == pytest.approx(sum(s[0] for s in singles), rel=1e-12)
    np.testing.assert_allclose(g, np.sum([s[1] for s in singles], axis=0), rtol=1e-9,
                               atol=1e-12 * np.max(np.abs(g)))
    K = so.sum_kmat(terms, X, white=white) + np.diag(e2)
    np.testing.assert_allclose(K @ A, Y, atol=1e-9)


# ---- host validation -------------------------------------------------------------------------------------------------
def _gp(**kw):
    import treegp_b200 as treegp

    kw.setdefault("optimizer", "none")
    return treegp.GPInterpolation(kernel="2.0 * RBF(1.0)", normalize=True, **kw)


def test_two_dimensional_y_validation_without_a_gpu():
    X, Y, e2 = _data(2, 3)
    with pytest.raises(ValueError, match="shape"):
        _gp().initialize(X, Y, y_err=np.sqrt(e2)[:, None] * np.ones((1, 3)))   # per-output errors
    with pytest.raises(ValueError, match="8"):
        _gp().initialize(X, np.zeros((len(X), 9)))
    for opt in ("two-pcf", "anisotropic"):
        gp = _gp(optimizer=opt)
        gp.initialize(X, Y, y_err=np.sqrt(e2))
        with pytest.raises(ValueError, match="1-D y"):
            gp.solve()
        with pytest.raises(ValueError, match="1-D y"):
            gp.return_2pcf()
    # normalize: one mean per output, no device needed
    gp = _gp()
    gp.initialize(X, Y, y_err=np.sqrt(e2))
    np.testing.assert_allclose(gp._mean, Y.mean(axis=0))
    assert gp._spatial_average.shape == Y.shape


def test_indice_meanify_with_several_outputs(tmp_path):
    from treegp_b200 import fitstable

    X, Y, _ = _data(2, 2)
    path = str(tmp_path / "mean.fits")
    grid = np.random.default_rng(4).uniform(0, 5, size=(30, 2))
    fitstable.write_table(path, {"COORDS0": grid[None], "PARAMS0": np.ones((1, 30, 4))})
    for bad in (None, 1, [0], [0, 1, 2], [0, 7], [0.0, 1.0]):
        with pytest.raises(ValueError, match="indice_meanify|columns"):
            _gp(average_fits=path, indice_meanify=bad).initialize(X, Y)


def test_multi_entry_points_reject_bad_arguments_without_a_gpu():
    """r outside 1 .. TGP_MAX_RHS and a bad descriptor are refused with -1 before any CUDA call."""
    from treegp_b200 import _cabi
    from treegp_b200._cabi import TgpKernelSum

    lib = _cabi.load()
    A16 = ctypes.c_void_p(16)
    ok = TgpKernelSum()
    ok.nterms, ok.ndim, ok.white = 1, 2, 0.0
    ok.term[0].family, ok.term[0].ndim, ok.term[0].amp = 0, 2, 1.0
    ok.term[0].m00, ok.term[0].m11 = 1.0, 1.0
    bad = TgpKernelSum()
    bad.nterms, bad.ndim = 0, 2
    calls = {
        "tgp_loglike_multi": lambda d, r: lib.tgp_loglike_multi(A16, A16, r, A16, 1000, ctypes.byref(d), A16, 1000, A16,
                                                                1, A16, A16, None, 0, None),
        "tgp_loglike_grad_multi": lambda d, r: lib.tgp_loglike_grad_multi(A16, A16, r, A16, 1000, ctypes.byref(d), A16,
                                                                          1000, A16, A16, A16, None, 0, A16, None),
        "tgp_predict_mean_multi": lambda d, r: lib.tgp_predict_mean_multi(A16, 10, A16, 1000, ctypes.byref(d), A16, r,
                                                                          A16, None),
        "tgp_predict_mean_trunc_multi": lambda d, r: lib.tgp_predict_mean_trunc_multi(A16, 10, A16, 1000,
                                                                                      ctypes.byref(d), A16, r, A16,
                                                                                      A16, None),
    }
    for name, call in calls.items():
        for r in (0, 9, -1):
            assert call(ok, r) == -1, (name, r)
            assert b"TGP_MAX_RHS" in lib.tgp_last_error(), name
        assert call(bad, 2) == -1, name
        assert b"kernel sum descriptor" in lib.tgp_last_error(), name
    assert lib.tgp_loglike_grad_multi_work_doubles(1000, 1, 0) == -1
    assert lib.tgp_loglike_grad_multi_work_doubles(1000, 1, 9) == -1
    assert lib.tgp_loglike_grad_multi_work_doubles(1000, 2, 4) == lib.tgp_loglike_grad_sum_work_doubles(1000, 2)
