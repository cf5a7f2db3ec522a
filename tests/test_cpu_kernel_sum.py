"""CPU: sum kernels without a GPU -- lowering of scikit-learn Sum trees (kernels.lower_kernel_sum, kernels.lower), the
chain rule to sklearn's theta (lower_kernel_sum_jacobian), the numpy sum oracle against scikit-learn's own
GaussianProcessRegressor, the support cut-off of a sum and the envelope decision it drives, and argument validation of
the *_sum C entry points."""
import ctypes

import numpy as np
import pytest

import sum_oracle as so


def _kernel(s):
    from treegp_b200 import eval_kernel

    return eval_kernel(s)


def _params(desc):
    """(ln amp_c, m00_c, m01_c, m11_c for every term, ln white) of a TgpKernelSum."""
    p = []
    for c in range(desc.nterms):
        t = desc.term[c]
        p += [np.log(t.amp), t.m00, t.m01, t.m11]
    return np.array(p + [np.log(desc.white) if desc.white > 0 else 0.0])


VK2 = "AnisotropicVonKarman(invLam=array([[0.5, 0.1], [0.1, 0.4]]))"
RBF2 = "AnisotropicRBF(invLam=array([[0.9, -0.35], [-0.35, 0.6]]))"


# ---- lowering ------------------------------------------------------------------------------------------------------
def test_accepted_trees_distribute_constants_and_add_white_levels():
    from treegp_b200 import _cabi
    from treegp_b200.kernels import lower, lower_kernel_sum

    d = lower_kernel_sum(_kernel("4.0 * %s + 0.5 * RBF(20.0) + WhiteKernel(1e-3)" % VK2), 2)
    assert isinstance(d, _cabi.TgpKernelSum) and d.nterms == 2 and d.ndim == 2 and d.white == 1e-3
    assert [d.term[c].family for c in range(2)] == [_cabi.FAM_VONKARMAN, _cabi.FAM_RBF]   # tree order
    assert [d.term[c].amp for c in range(2)] == [4.0, 0.5]
    assert (d.term[0].m00, d.term[0].m01, d.term[0].m11) == (0.5, 0.1, 0.4)
    assert d.term[1].m00 == pytest.approx(1 / 400.0, rel=1e-15) and d.term[1].m01 == 0.0

    # c * (a + b) -> c a + c b; scaled and repeated WhiteKernels add up
    d = lower_kernel_sum(_kernel("2.0 * (3.0 * RBF(1.0) + Matern(0.5, nu=1.5) + WhiteKernel(0.1)) + WhiteKernel(0.2)"),
                         1)
    assert d.nterms == 2 and [d.term[c].amp for c in range(2)] == [6.0, 2.0]
    assert d.term[1].family == _cabi.FAM_MATERN32 and d.white == pytest.approx(0.4, rel=1e-15)
    assert d.term[0].ndim == d.term[1].ndim == 1

    # no white level; four terms is the limit
    d = lower_kernel_sum(_kernel("RBF(1.0) + VonKarman(2.0) + Matern(1.0, nu=0.5) + Matern(1.0, nu=2.5)"), 2)
    assert d.nterms == 4 and d.white == 0.0
    assert [d.term[c].family for c in range(4)] == [0, 1, 2, 4]

    # the dispatcher keeps every single-term kernel on the single-term descriptor
    assert isinstance(lower(_kernel("2.0 * RBF(0.8)"), 2), _cabi.TgpKernel)
    assert isinstance(lower(_kernel("ConstantKernel(2.0) * (ConstantKernel(0.5) * RBF([1.0, 0.4]))"), 2), _cabi.TgpKernel)
    assert isinstance(lower(_kernel("RBF(0.8) + WhiteKernel(0.1)"), 2), _cabi.TgpKernelSum)


@pytest.mark.parametrize("kstr,what", [
    ("RBF(1.0) * Matern(1.0) + WhiteKernel(0.1)", "more than one non-constant factor"),
    ("(RBF(1.0) + WhiteKernel(0.1)) * (RBF(2.0) + WhiteKernel(0.1))", "more than one non-constant factor"),
    ("RBF(1.0) + ConstantKernel(2.0)", "constant offset"),
    ("RBF(1.0) + DotProduct(1.0)", "DotProduct"),
    ("RBF(1.0) + Matern(1.0, nu=0.7)", "Matern"),
    ("WhiteKernel(0.1)", "no stationary term"),
    ("2.0 * WhiteKernel(0.1) + WhiteKernel(0.2)", "no stationary term"),
    ("RBF(1.0) + RBF(2.0) + RBF(3.0) + RBF(4.0) + RBF(5.0)", "5 stationary terms"),
])
def test_rejected_trees_name_the_offending_term(kstr, what):
    from treegp_b200 import _cabi
    from treegp_b200.kernels import lower, lower_kernel_sum, lower_kernel_sum_jacobian

    for fn in (lower_kernel_sum, lower_kernel_sum_jacobian, lower):
        with pytest.raises(_cabi.TgpError, match=what):
            fn(_kernel(kstr), 2)


def test_term_dimension_must_match_the_coordinates():
    from treegp_b200.kernels import lower_kernel_sum

    with pytest.raises(ValueError):
        lower_kernel_sum(_kernel("%s + WhiteKernel(0.1)" % RBF2), 1)
    with pytest.raises(ValueError):
        lower_kernel_sum(_kernel("RBF([1.0, 2.0, 3.0]) + WhiteKernel(0.1)"), 2)


SUMS = [
    ("4.0 * %s + 0.5 * RBF(20.0) + WhiteKernel(1e-3)" % VK2, 2),
    ("ConstantKernel(2.0) * %s + ConstantKernel(0.3) * %s + WhiteKernel(0.01)" % (RBF2, VK2), 2),
    ("ConstantKernel(2.0) * (RBF([0.7, 1.3]) + ConstantKernel(0.5) * Matern(0.6, nu=2.5)) + WhiteKernel(0.05)", 2),
    ("RBF(0.8) + WhiteKernel(0.1) + 3.0 * WhiteKernel(0.02)", 1),
    ("ConstantKernel(3.0, 'fixed') * %s + RBF(0.8, length_scale_bounds='fixed') + WhiteKernel(0.1, 'fixed')" % VK2, 2),
    ("VonKarman(0.9) + ConstantKernel(0.2) * Matern(1.5, nu=0.5) * ConstantKernel(2.0)", 2),
]


@pytest.mark.parametrize("kstr,ndim", SUMS)
def test_sum_jacobian_against_central_differences(kstr, ndim):
    from treegp_b200.kernels import lower_kernel_sum, lower_kernel_sum_jacobian

    k = _kernel(kstr)
    desc, J = lower_kernel_sum_jacobian(k, ndim)
    np.testing.assert_array_equal(_params(desc), _params(lower_kernel_sum(k, ndim)))
    theta = np.array(k.theta, dtype=float)
    assert J.shape == (4 * desc.nterms + 1, len(theta))
    h = 1e-6
    for j in range(len(theta)):
        e = np.zeros_like(theta)
        e[j] = h
        fd = (_params(lower_kernel_sum(k.clone_with_theta(theta + e), ndim))
              - _params(lower_kernel_sum(k.clone_with_theta(theta - e), ndim))) / (2 * h)
        np.testing.assert_allclose(J[:, j], fd, rtol=1e-7, atol=1e-8 * max(1.0, np.max(np.abs(fd))))
    if desc.white == 0.0:
        assert np.all(J[-1] == 0.0)


def test_fixed_hyperparameters_have_no_column():
    from treegp_b200.kernels import lower_kernel_sum_jacobian

    _, J = lower_kernel_sum_jacobian(_kernel(SUMS[4][0]), 2)
    assert J.shape == (9, 3)       # only the von Karman metric's three thetas are free
    assert np.all(J[0] == 0.0) and np.all(J[4:] == 0.0)


# ---- the oracle --------------------------------------------------------------------------------------------------
SKLEARN_SUMS = [
    ("ConstantKernel(2.0) * RBF(0.7) + ConstantKernel(0.5) * Matern(1.3, nu=1.5) + WhiteKernel(0.05)", 2),
    ("ConstantKernel(1.5) * (RBF([0.6, 1.1]) + Matern(0.4, nu=0.5)) + WhiteKernel(0.02) + WhiteKernel(0.03)", 2),
    ("ConstantKernel(0.8) * Matern(0.5, nu=2.5) + RBF(2.0) + WhiteKernel(0.1)", 1),
    ("ConstantKernel(3.0, 'fixed') * RBF(0.9) + ConstantKernel(0.4) * RBF(3.0, length_scale_bounds='fixed')", 2),
]


@pytest.mark.parametrize("kstr,ndim", SKLEARN_SUMS)
def test_oracle_against_sklearn_gaussian_process_regressor(kstr, ndim):
    """sklearn's GaussianProcessRegressor(kernel, alpha=y_err**2).log_marginal_likelihood(theta, eval_gradient=True)
    is the reference's formula (kernel(X) + eye * y_err**2) with its own theta gradient."""
    from sklearn.gaussian_process import GaussianProcessRegressor
    from treegp_b200.kernels import lower_kernel_sum_jacobian

    rng = np.random.default_rng(3 + ndim)
    n = 140
    X = rng.uniform(0, 5, size=(n, ndim))
    X[7] = X[3]                                  # a duplicated point
    y = rng.normal(size=n)
    e2 = rng.uniform(0.01, 0.03, size=n)
    k = _kernel(kstr)
    gpr = GaussianProcessRegressor(kernel=k, alpha=e2, optimizer=None).fit(X, y)
    ref, ref_g = gpr.log_marginal_likelihood(k.theta, eval_gradient=True)
    desc, J = lower_kernel_sum_jacobian(k, ndim)
    terms, white = so.terms_of(desc)
    logl, g = so.sum_log_likelihood_gradient(terms, white, X, y, e2)
    assert logl == pytest.approx(ref, rel=1e-10)
    np.testing.assert_allclose(J.T @ g, ref_g, rtol=1e-7, atol=1e-8 * np.max(np.abs(ref_g)))


@pytest.mark.parametrize("ndim", [1, 2])
def test_oracle_gradient_against_central_differences(ndim):
    """Von Karman terms (not in sklearn) and the per-term coincident-point rule, with duplicated points."""
    rng = np.random.default_rng(11 + ndim)
    n = 150
    X = rng.uniform(0, 6, size=(n, ndim))
    X[10:14] = X[20:24]
    y = rng.normal(size=n)
    e2 = rng.uniform(0.01, 0.05, size=n)
    e2[10:14] += 2.0    # the von Karman rule between coincident points lowers K(X, X) by up to amp there
    e2[20:24] += 2.0
    M1 = np.array([[1.3]]) if ndim == 1 else np.array([[1.1, 0.3], [0.3, 0.7]])
    M2 = np.array([[0.2]]) if ndim == 1 else np.array([[0.25, -0.05], [-0.05, 0.15]])

    def flat(M):
        return [M[0, 0], 0.0, 0.0] if ndim == 1 else [M[0, 0], M[0, 1], M[1, 1]]

    p0 = np.array([np.log(1.7)] + flat(M1) + [np.log(0.6)] + flat(M2) + [np.log(0.04)])

    def unpack(p):
        def m(a):
            return np.array([[a[0]]]) if ndim == 1 else np.array([[a[0], a[1]], [a[1], a[2]]])
        return [("vonkarman", np.exp(p[0]), m(p[1:4])), ("rbf", np.exp(p[4]), m(p[5:8]))], np.exp(p[8])

    terms, white = unpack(p0)
    K = so.sum_kmat(terms, X, white=white)
    assert K[10, 20] == pytest.approx(0.6)           # the RBF term keeps its amplitude between coincident points
    logl, g = so.sum_log_likelihood_gradient(terms, white, X, y, e2)
    for j in range(9):
        if ndim == 1 and j in (2, 3, 6, 7):
            assert g[j] == 0.0
            continue
        e = np.zeros(9)
        e[j] = 1e-5
        fd = (so.sum_log_likelihood_gradient(*unpack(p0 + e), X, y, e2)[0]
              - so.sum_log_likelihood_gradient(*unpack(p0 - e), X, y, e2)[0]) / 2e-5
        assert abs(g[j] - fd) <= 1e-5 * max(1.0, np.max(np.abs(g))), (j, g[j], fd)


# ---- cut-offs and the envelope decision ----------------------------------------------------------------------------
def test_support_cutoffs_of_a_sum_are_the_per_axis_maximum():
    from treegp_b200 import backend
    from treegp_b200.kernels import lower_kernel, lower_kernel_sum

    s = "0.5 * AnisotropicRBF(invLam=array([[4.0, 0.0], [0.0, 0.01]])) + 2.0 * %s + WhiteKernel(0.1)" % VK2
    d = lower_kernel_sum(_kernel(s), 2)
    a = backend.support_cutoffs(d.term[0])
    b = backend.support_cutoffs(d.term[1])
    assert backend.support_cutoffs(d) == [max(a[0], b[0]), max(a[1], b[1])]
    assert backend.support_cutoffs(lower_kernel(_kernel("2.0 * %s" % VK2), 2)) == b
    bad = lower_kernel_sum(_kernel("RBF(1.0) + RBF(2.0)"), 2)
    bad.term[1].m11 = -1.0
    assert np.isnan(backend.support_cutoffs(bad)[1])


def test_plan_envelope_for_sums():
    """The envelope serves the union of the supports: a short term alone bands, a long-range term in the sum keeps
    the dense path, and the white level changes nothing."""
    import torch
    from treegp_b200 import backend
    from treegp_b200.kernels import lower_kernel, lower_kernel_sum

    rng = np.random.default_rng(0)
    X = torch.as_tensor(rng.uniform(0, 160.0, size=(8000, 2)))
    short = "2.0 * AnisotropicVonKarman(invLam=array([[0.5, 0.1], [0.1, 0.4]]))"
    p1 = backend.plan_envelope(X, lower_kernel(_kernel(short), 2))
    p2 = backend.plan_envelope(X, lower_kernel_sum(_kernel(short + " + WhiteKernel(0.01)"), 2))
    assert p1 is not None and p2 is not None
    assert p1["axis"] == p2["axis"] and p1["dcut"] == p2["dcut"]
    np.testing.assert_array_equal(p1["row_end"], p2["row_end"])
    p3 = backend.plan_envelope(X, lower_kernel_sum(_kernel(short + " + 0.1 * RBF(3.0)"), 2))
    assert p3 is not None and p3["dcut"] > p1["dcut"] and p3["flops"] > p1["flops"]
    assert backend.plan_envelope(X, lower_kernel_sum(_kernel(short + " + 0.1 * RBF(60.0)"), 2)) is None


# ---- C ABI validation --------------------------------------------------------------------------------------------
def _sum_desc(nterms=2, ndim=2, white=0.1, families=(0, 1)):
    from treegp_b200 import _cabi

    d = _cabi.TgpKernelSum()
    d.nterms, d.ndim, d.white = nterms, ndim, white
    for c in range(_cabi.MAX_TERMS):
        d.term[c] = _cabi.TgpKernel(families[c % len(families)], ndim, 1.0, 1.0, 0.0, 1.0)
    return d


def _bad_descs():
    bad = {"nterms 0": _sum_desc(nterms=0), "nterms 5": _sum_desc(nterms=5), "negative white": _sum_desc(white=-1e-3),
           "nan white": _sum_desc(white=float("nan")), "inf white": _sum_desc(white=float("inf")),
           "bad family": _sum_desc(families=(0, 9)), "ndim 3": _sum_desc(ndim=3)}
    d = _sum_desc()
    d.term[1].ndim = 1
    bad["mismatched ndim"] = d
    return bad


def test_sum_entry_points_reject_bad_descriptors_without_a_gpu():
    """Argument validation happens before any CUDA call; entries past nterms are not read."""
    from treegp_b200 import _cabi

    lib = _cabi.load()
    A16 = ctypes.c_void_p(16)
    re2 = np.array([1000, 1000], dtype=np.int64)
    rep = ctypes.c_void_p(re2.ctypes.data)
    calls = {
        "tgp_kmat_sym_sum": lambda d: lib.tgp_kmat_sym_sum(A16, 1000, ctypes.byref(d), None, A16, 1000, 1, None),
        "tgp_kmat_cross_sum": lambda d: lib.tgp_kmat_cross_sum(A16, 10, A16, 1000, ctypes.byref(d), A16, 1000, None),
        "tgp_loglike_sum": lambda d: lib.tgp_loglike_sum(A16, A16, A16, 1000, ctypes.byref(d), A16, 1000, A16, 1, A16,
                                                         A16, rep, 2, None),
        "tgp_loglike_grad_sum": lambda d: lib.tgp_loglike_grad_sum(A16, A16, A16, 1000, ctypes.byref(d), A16, 1000,
                                                                   A16, A16, A16, rep, 2, A16, None),
        "tgp_predict_mean_sum": lambda d: lib.tgp_predict_mean_sum(A16, 10, A16, 1000, ctypes.byref(d), A16, A16, None),
        "tgp_predict_mean_trunc_sum": lambda d: lib.tgp_predict_mean_trunc_sum(A16, 10, A16, 1000, ctypes.byref(d),
                                                                               A16, A16, A16, None),
        "tgp_predict_var_sum": lambda d: lib.tgp_predict_var_sum(A16, 10, A16, 1000, ctypes.byref(d), A16, 1000, rep,
                                                                 2, A16, 128, A16, None),
    }
    for name, call in calls.items():
        for what, d in _bad_descs().items():
            assert call(d) == -1, (name, what)
            assert b"kernel sum descriptor" in lib.tgp_last_error(), (name, what)
    ok = _sum_desc(nterms=1)
    ok.term[1].family = 99          # past nterms: not read
    assert lib.tgp_loglike_sum(A16, A16, A16, 1000, ctypes.byref(ok), A16, 1000, A16, 1, A16, A16, rep, 3, None) == -1
    assert b"row_end" in lib.tgp_last_error()
    assert lib.tgp_loglike_grad_sum(A16, A16, A16, 1000, ctypes.byref(ok), A16, 1000, A16, A16, A16, rep, 2, None,
                                    None) == -1
    assert b"scratch" in lib.tgp_last_error()
    assert lib.tgp_loglike_grad_sum_work_doubles(1000, 0) == -1
    assert lib.tgp_loglike_grad_sum_work_doubles(1000, 5) == -1
    assert lib.tgp_loglike_grad_sum_work_doubles(1000, 1) == lib.tgp_selinv_work_doubles(1000)   # selinv dominates
    n = 10 ** 6                     # here the 17 partials per 64 x 64 tile dominate
    nt = -(-n // 64)
    assert lib.tgp_loglike_grad_sum_work_doubles(n, 4) >= 17 * nt * (nt + 1) // 2
