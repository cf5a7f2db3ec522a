"""GPU parity: the envelope (variable-band) forms of the dense calls -- tgp_potrf_env, tgp_loglike_env,
tgp_trsm_rows_env, tgp_predict_var_env -- against the dense calls they restrict (csrc/dense.cu, csrc/predict.cu)
and against the oracle, and the host logic that chooses them (backend.plan_envelope, GPInterpolation.BANDED_SOLVE,
log_likelihood.BANDED).  The reference factorises the dense matrix whatever the kernel (gp_interp.py:181,
log_likelihood.py:30); with the points sorted along one axis and a kernel below 1e-40 of its amplitude beyond d_cut
the two give the same numbers to rounding."""
import numpy as np
import pytest

from oracle import gp_oracle as go

pytestmark = pytest.mark.gpu

MI = np.array([[0.9, -0.35], [-0.35, 0.6]])
KSTR = {"rbf2": "2.0 * AnisotropicRBF(invLam=array([[0.9, -0.35], [-0.35, 0.6]]))",
        "vk2": "2.0 * AnisotropicVonKarman(invLam=array([[0.9, -0.35], [-0.35, 0.6]]))",
        "rbf1": "2.0 * RBF(0.8)"}


def _problem(case, n, field, seed=23):
    from treegp_b200 import backend, eval_kernel
    from treegp_b200.kernels import lower_kernel

    rng = np.random.default_rng(seed)
    ndim = 1 if case == "rbf1" else 2
    X = rng.uniform(0, field, size=(n, ndim))
    desc = lower_kernel(eval_kernel(KSTR[case]), ndim)
    y = rng.normal(size=n)
    e2 = rng.uniform(0.005, 0.02, size=n)
    plan = backend.plan_envelope(backend.as_points(X), desc)
    return X, y, e2, desc, plan


@pytest.mark.parametrize("case,n,field", [("rbf2", 6000, 260.0), ("vk2", 4500, 300.0), ("rbf1", 5000, 900.0),
                                          ("rbf2", 4100, 120.0)])
def test_potrf_env_and_loglike_env_equal_the_dense_calls(gpu_ready, case, n, field):
    from treegp_b200 import backend

    X, y, e2, desc, plan = _problem(case, n, field)
    assert plan is not None and plan["flops"] * 2 <= plan["flops_dense"]
    o = plan["order"]
    Xs = backend.as_points(X)[o].contiguous()
    ys, es = backend.to_device(y)[o].contiguous(), backend.to_device(e2)[o].contiguous()
    re = plan["row_end"]
    assert re.dtype == np.int64 and len(re) == (n + 511) // 512 and re[-1] == n and np.all(np.diff(re) >= 0)
    # factor
    A = backend.kmat_sym(Xs, desc, es, lower_only=True)
    B = A.clone()
    assert int(backend.potrf(A, n).item()) == 0 and int(backend.potrf(B, n, row_end=re).item()) == 0
    La, Lb = np.tril(A[:, :n].cpu().numpy()), np.tril(B[:, :n].cpu().numpy())
    assert np.max(np.abs(La - Lb)) <= 1e-11 * np.max(np.abs(La))
    # outside the envelope the dense factor is (numerically) zero and the envelope factor was never touched
    outside = np.zeros((n, n), dtype=bool)
    for b, r in enumerate(re):
        outside[r:, 512 * b:512 * (b + 1)] = True
    assert outside.any() and np.max(np.abs(La[outside])) < 1e-30 and np.max(np.abs(Lb[outside])) < 1e-30
    # whole likelihood evaluation, with and without the backward sweep
    for want_alpha in (False, True):
        d_out, d_info, d_alpha, _ = backend.loglike(Xs, ys, es, desc, want_alpha=want_alpha)
        e_out, e_info, e_alpha, _ = backend.loglike(Xs, ys, es, desc, want_alpha=want_alpha, row_end=re)
        assert int(d_info.item()) == 0 and int(e_info.item()) == 0
        np.testing.assert_allclose(e_out.cpu().numpy(), d_out.cpu().numpy(), rtol=1e-11)
        da = d_alpha.cpu().numpy()
        np.testing.assert_allclose(e_alpha.cpu().numpy(), da, rtol=0, atol=1e-9 * np.max(np.abs(da)))
    # and the oracle (scipy) on the unsorted problem
    fam = "vonkarman" if case == "vk2" else "rbf"
    kw = dict(amp=2.0, invLam=np.array([[1.0 / 0.64]])) if case == "rbf1" else dict(amp=2.0, invLam=MI)
    logl, alpha = go.log_likelihood(go.kmat(fam, X, **kw) + np.diag(e2), y)
    assert abs(float(e_out[0].item()) - logl) <= 1e-10 * abs(logl)
    got = np.empty(n)
    got[o.cpu().numpy()] = e_alpha.cpu().numpy()
    np.testing.assert_allclose(got, alpha, rtol=0, atol=1e-8 * np.max(np.abs(alpha)))


def test_potrf_env_carries_extra_rows_as_the_dense_call(gpu_ready):
    """tgp_potrf_env with right-hand-side rows below the matrix (nrows > 0): the factor and the rows L^-1 y equal
    those of tgp_potrf_rows on the same sorted problem.  The rows ride inside the panel solves of the block columns
    whose envelope reaches N and take their own solve and update in the others."""
    import torch
    from treegp_b200 import _cabi, backend

    n, r = 6000, 3
    X, y, e2, desc, plan = _problem("rbf2", n, 260.0)
    o, re = plan["order"], plan["row_end"]
    assert re[0] < n and re[-1] == n
    A = backend.alloc_matrix(n + r, n)
    backend.kmat_sym(backend.as_points(X)[o].contiguous(), desc, backend.to_device(e2)[o].contiguous(), out=A,
                     lower_only=True)
    A[n:, :n] = backend.to_device(np.random.default_rng(5).normal(size=(r, n)))
    B = A.clone()
    lib = _cabi.load()
    ia, ib = (torch.ones(1, dtype=torch.int32, device=A.device) for _ in range(2))
    assert lib.tgp_potrf_rows(backend._p(A), n, A.stride(0), r, backend._p(ia), backend._stream()) == 0
    assert lib.tgp_potrf_env(backend._p(B), n, B.stride(0), backend._host_i64(re), len(re), r, backend._p(ib),
                             backend._stream()) == 0
    assert int(ia.item()) == 0 and int(ib.item()) == 0
    La, Lb = np.tril(A[:n, :n].cpu().numpy()), np.tril(B[:n, :n].cpu().numpy())
    assert np.max(np.abs(La - Lb)) <= 1e-11 * np.max(np.abs(La))
    Wa, Wb = A[n:, :n].cpu().numpy(), B[n:, :n].cpu().numpy()
    assert np.max(np.abs(Wa - Wb)) <= 1e-11 * np.max(np.abs(Wa))


def test_envelope_reports_a_matrix_that_is_not_positive_definite(gpu_ready):
    """info is the failing leading minor, as from the dense call, and logL is -inf (log_likelihood.py:38-39)."""
    from treegp_b200 import backend

    X, y, e2, desc, plan = _problem("rbf2", 5000, 240.0)
    o = plan["order"]
    Xs = backend.as_points(X)[o].contiguous()
    e2 = e2.copy()
    e2[3210] = -50.0
    ys, es = backend.to_device(y)[o].contiguous(), backend.to_device(e2).contiguous()
    d_out, d_info, _, _ = backend.loglike(Xs, ys, es, desc)
    e_out, e_info, _, _ = backend.loglike(Xs, ys, es, desc, row_end=plan["row_end"])
    assert int(d_info.item()) == int(e_info.item()) > 0
    assert float(e_out[0].item()) == -np.inf and float(d_out[0].item()) == -np.inf
    # the sweeps that follow the failed factorisation run on NaNs: they must pass through, not wait for ever
    _, a_info, _, _ = backend.loglike(Xs, ys, es, desc, want_alpha=True, row_end=plan["row_end"])
    assert int(a_info.item()) == int(e_info.item())
    from treegp_b200 import _cabi
    assert _cabi.load().tgp_device_error(0) == 0


@pytest.mark.parametrize("case", ["rbf2", "vk2"])
def test_trsm_rows_env_and_predict_var_env(gpu_ready, case):
    from treegp_b200 import backend

    n, m, field = 5200, 3000, 280.0
    X, y, e2, desc, plan = _problem(case, n, field)
    o, re = plan["order"], plan["row_end"]
    Xs = backend.as_points(X)[o].contiguous()
    L = backend.kmat_sym(Xs, desc, backend.to_device(e2)[o].contiguous(), lower_only=True)
    assert int(backend.potrf(L, n, row_end=re).item()) == 0
    rng = np.random.default_rng(1)
    Xt = rng.uniform(0, field, size=(m, 2))
    V1 = backend.kmat_cross(Xt, Xs, desc)
    V2 = V1.clone()
    backend.trsm_rows(L, n, V1, m)
    backend.trsm_rows(L, n, V2, m, row_end=re)
    a, b = V1[:, :n].cpu().numpy(), V2[:, :n].cpu().numpy()
    assert np.max(np.abs(a - b)) <= 1e-11 * np.max(np.abs(a))
    v1 = backend.predict_var(Xt, Xs, desc, L, chunk=1024).cpu().numpy()
    v2 = backend.predict_var(Xt, Xs, desc, L, chunk=1024, row_end=re).cpu().numpy()
    np.testing.assert_allclose(v2, v1, rtol=0, atol=1e-11)
    # a trailing sub-system with its own envelope (what the windowed variance solves)
    s = 1216
    re_s = backend.envelope_rows(plan["x"], plan["dcut"], start=s)
    v3 = backend.predict_var(Xt[:500], Xs[s:], desc, L[s:, s:], chunk=512).cpu().numpy()
    v4 = backend.predict_var(Xt[:500], Xs[s:], desc, L[s:, s:], chunk=512, row_end=re_s).cpu().numpy()
    np.testing.assert_allclose(v4, v3, rtol=0, atol=1e-11)


def test_gpinterpolation_banded_solve_equals_dense_solve(gpu_ready):
    """Public class: same alpha (in the caller's order), mean, covariance and variance with the envelope
    factorisation (the default when it pays) and with the dense one."""
    import treegp_b200 as treegp

    rng = np.random.default_rng(4)
    n, field = 5000, 250.0
    X = rng.uniform(0, field, size=(n, 2))
    y = rng.normal(size=n)
    yerr = rng.uniform(0.05, 0.15, size=n)
    Xt = rng.uniform(0, field, size=(7000, 2))
    res = []
    for banded in (True, False):
        gp = treegp.GPInterpolation(kernel=KSTR["vk2"], optimizer="none", normalize=True)
        gp.BANDED_SOLVE, gp.VAR_CHUNK = banded, 1024
        gp.initialize(X, y, y_err=yerr)
        mean = gp.predict(Xt)
        assert (gp._envelope is not None) == banded
        m2, cov = gp.predict(Xt[:300], return_cov=True)
        _, var = gp.predict_var(Xt)
        gp.WINDOWED_VARIANCE = False
        _, var_plain = gp.predict_var(Xt[:1500])
        res.append((gp._alpha.copy(), mean, cov, var, var_plain))
    (a1, m1, c1, v1, p1), (a0, m0, c0, v0, p0) = res
    np.testing.assert_allclose(a1, a0, rtol=0, atol=1e-9 * np.max(np.abs(a0)))
    np.testing.assert_allclose(m1, m0, rtol=0, atol=1e-9)
    np.testing.assert_allclose(c1, c0, rtol=0, atol=1e-10)
    np.testing.assert_allclose(v1, v0, rtol=0, atol=1e-10)
    np.testing.assert_allclose(p1, p0, rtol=0, atol=1e-10)
    np.testing.assert_allclose(v1[:1500], p1, rtol=0, atol=1e-10)
    np.testing.assert_allclose(np.diag(c1), v1[:300], rtol=0, atol=1e-10)


def test_log_likelihood_search_with_and_without_the_envelope(gpu_ready):
    """log_likelihood.log_likelihood: the same value at fixed kernels (1e-11), and the L-BFGS-B fit
    (log_likelihood.py:43-62) ends at the same maximum."""
    import treegp_b200 as treegp
    from treegp_b200.two_pcf import get_correlation_length_matrix

    rng = np.random.default_rng(12)
    n, field = 4500, 70.0
    inv = np.linalg.inv(get_correlation_length_matrix(0.5, 0.2, 0.2))
    kstr = "4.0 * AnisotropicRBF(invLam=array([[%.17g, %.17g], [%.17g, %.17g]]))" % (inv[0, 0], inv[0, 1], inv[1, 0], inv[1, 1])
    X = rng.uniform(-field / 2, field / 2, size=(n, 2))
    kern = treegp.eval_kernel(kstr)
    y, y_err = treegp.sample_grf(kern, X, noise=0.05, seed=3)
    vals = {}
    for banded in (True, False):
        ll = treegp.log_likelihood(X, y, y_err)
        ll.BANDED = banded
        vals[banded] = [ll.log_likelihood(kern.clone_with_theta(kern.theta + d)) for d in (0.0, 0.3, -0.4)]
        assert (getattr(ll, "n_banded_evaluations", 0) == 3) == banded
    np.testing.assert_allclose(vals[True], vals[False], rtol=1e-11)
    fits = {}
    for banded in (True, False):
        ll = treegp.log_likelihood(X, y, y_err)
        ll.BANDED = banded
        start = kern.clone_with_theta(kern.theta + np.array([0.2, -0.2, 0.1, 0.1]))
        k = ll.optimizer(start)
        fits[banded] = (np.array(k.theta), ll._logL, ll.n_evaluations)
    assert abs(fits[True][1] - fits[False][1]) <= 1e-7 * abs(fits[False][1])
    np.testing.assert_allclose(fits[True][0], fits[False][0], rtol=0, atol=5e-3)
