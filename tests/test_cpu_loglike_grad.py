"""CPU: the pieces of the analytic log-likelihood gradient that need no GPU -- the host chain rule
(kernels.lower_kernel_jacobian), the profile derivatives f'(q) of csrc/profile_dq.cuh compiled for the host, the numpy
oracle of the gradient, the blocked selected-inverse recurrence that tgp_selinv runs, and argument validation of the
two new C entry points."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from oracle import gp_oracle as go
import grad_oracle as gro

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

KERNELS = [
    ("2.0 * RBF(0.8)", 1), ("2.0 * RBF(0.8)", 2), ("RBF([0.7, 1.3])", 2),
    ("1.5 * Matern(length_scale=0.6, nu=0.5)", 2), ("Matern(length_scale=0.6, nu=1.5)", 1),
    ("0.7 * Matern(length_scale=[0.6, 1.1], nu=2.5)", 2), ("Matern(length_scale=2.0, nu=np.inf)", 2),
    ("3.0 * VonKarman(0.9)", 2), ("VonKarman(0.9)", 1), ("VonKarman([0.9, 1.7])", 2),
    ("4.0 * AnisotropicRBF(invLam=array([[0.9, -0.35], [-0.35, 0.6]]))", 2),
    ("AnisotropicVonKarman(invLam=array([[0.5, 0.1], [0.1, 0.4]])) * 2.5", 2),
    ("AnisotropicRBF(invLam=array([[1.7]]))", 1),
    ("ConstantKernel(2.0) * (ConstantKernel(0.5) * RBF([1.0, 0.4]))", 2),
    ("ConstantKernel(3.0, 'fixed') * AnisotropicVonKarman(invLam=array([[0.5, 0.1], [0.1, 0.4]]))", 2),
    ("ConstantKernel(3.0, 'fixed') * RBF(0.8, length_scale_bounds='fixed') * ConstantKernel(0.2)", 2),
]


def _kernel(s):
    from treegp_b200 import eval_kernel

    return eval_kernel(s.replace("np.inf", "float('inf')"))


def _params(desc):
    return np.array([np.log(desc.amp), desc.m00, desc.m01, desc.m11])


@pytest.mark.parametrize("kstr,ndim", KERNELS)
def test_lower_kernel_jacobian_against_central_differences(kstr, ndim):
    from treegp_b200.kernels import lower_kernel, lower_kernel_jacobian

    k = _kernel(kstr)
    desc, J = lower_kernel_jacobian(k, ndim)
    np.testing.assert_array_equal(_params(desc), _params(lower_kernel(k, ndim)))
    theta = np.array(k.theta, dtype=float)
    assert J.shape == (4, len(theta))
    h = 1e-6
    for j in range(len(theta)):
        e = np.zeros_like(theta)
        e[j] = h
        fd = (_params(lower_kernel(k.clone_with_theta(theta + e), ndim))
              - _params(lower_kernel(k.clone_with_theta(theta - e), ndim))) / (2 * h)
        np.testing.assert_allclose(J[:, j], fd, rtol=1e-7, atol=1e-8 * max(1.0, np.max(np.abs(fd))))
    if ndim == 1:
        assert np.all(J[2:] == 0.0)


def test_fixed_hyperparameters_have_no_column_and_other_kernels_raise():
    from treegp_b200 import _cabi
    from treegp_b200.kernels import lower_kernel_jacobian

    _, J = lower_kernel_jacobian(_kernel("ConstantKernel(3.0, 'fixed') * RBF(0.8)"), 2)
    assert J.shape == (4, 1) and J[0, 0] == 0.0
    _, J = lower_kernel_jacobian(_kernel("ConstantKernel(3.0) * RBF(0.8, length_scale_bounds='fixed')"), 2)
    assert J.shape == (4, 1) and np.all(J[:, 0] == [1.0, 0.0, 0.0, 0.0])
    for bad in ("RBF(1.0) + WhiteKernel(0.1)", "RBF(1.0) * Matern(1.0)", "Matern(1.0, nu=0.7)"):
        with pytest.raises(_cabi.TgpError):
            lower_kernel_jacobian(_kernel(bad), 2)


# ---- f'(q): the device header compiled for the host ------------------------------------------------------------
@pytest.fixture(scope="module")
def dq_host(tmp_path_factory):
    d = tmp_path_factory.mktemp("dq")
    src = d / "h.cpp"
    src.write_text('#include "profile_dq.cuh"\nextern "C" void dq_eval(int fam, const double* q, long n, double* out)'
                   '{ for (long i = 0; i < n; i++) out[i] = tgp_profile_dq_family(fam, q[i], tgp_vk_phi_host); }\n'
                   'extern "C" void f_eval(const double* q, long n, double* out)'
                   '{ for (long i = 0; i < n; i++) out[i] = tgp_vk_profile(q[i], tgp_vk_phi_host); }\n')
    so = d / "libdq.so"
    subprocess.check_call(["/usr/bin/g++", "-O2", "-ffp-contract=off", "-shared", "-fPIC",
                           "-I", os.path.join(ROOT, "treegp_b200", "csrc"), str(src), "-o", str(so)])
    lib = ctypes.CDLL(str(so))

    def call(fn, *args):
        q = np.ascontiguousarray(args[-1], dtype=np.float64)
        out = np.empty_like(q)
        fn(*args[:-1], q.ctypes.data_as(ctypes.c_void_p), ctypes.c_long(q.size), out.ctypes.data_as(ctypes.c_void_p))
        return out

    return (lambda fam, q: call(lib.dq_eval, ctypes.c_int(fam), q)), (lambda q: call(lib.f_eval, q))


def test_vk_profile_derivative_against_mpmath(dq_host):
    import mpmath as mp
    from treegp_b200 import _cabi

    dq, _ = dq_host
    mp.mp.dps = 40
    c = mp.mpf(2) ** (mp.mpf(1) / 6) / mp.gamma(mp.mpf(5) / 6)
    rng = np.random.default_rng(2)
    d = np.concatenate([10 ** rng.uniform(-6, 1.2, 1500), rng.uniform(0, 3, 500),
                        [1 / (2 * np.pi), 0.5 / np.pi, 1.0 / np.pi, 2.0 / np.pi]])
    got = dq(_cabi.FAM_VONKARMAN, d * d)
    worst = 0.0
    for di, gi in zip(d, got):
        q = mp.mpf(float(di)) ** 2
        z = 2 * mp.pi * mp.sqrt(q)
        truth = -2 * mp.pi ** 2 * c * z ** (-mp.mpf(1) / 6) * mp.besselk(mp.mpf(1) / 6, z)
        err = abs(mp.mpf(float(gi)) - truth) / max(abs(truth), mp.mpf(1e-300))
        worst = max(worst, float(err))
    assert worst < 1e-11, worst
    assert dq(_cabi.FAM_VONKARMAN, np.array([1e6]))[0] == 0.0


@pytest.mark.parametrize("fam,name", [(0, "rbf"), (2, "matern12"), (3, "matern32"), (4, "matern52"), (1, "vonkarman")])
def test_profile_derivatives_against_numerical_derivatives(dq_host, fam, name):
    """Closed forms (and the von Karman one) against a central difference of the profile itself."""
    dq, vk_f = dq_host
    q = np.concatenate([10 ** np.linspace(-3, 2, 400), np.linspace(0.05, 30, 400)])
    h = 1e-6 * q
    if name == "vonkarman":
        fd = (vk_f(q + h) - vk_f(q - h)) / (2 * h)
    else:
        f = lambda x: go.kmat(name, np.sqrt(x)[:, None], np.zeros((1, 1)), length_scale=1.0)[:, 0]
        fd = (f(q + h) - f(q - h)) / (2 * h)
    got = dq(fam, q)
    np.testing.assert_allclose(got, fd, rtol=1e-6, atol=1e-9 * np.max(np.abs(fd)))
    np.testing.assert_allclose(got, gro.profile_dq(name, q), rtol=1e-9, atol=0)


# ---- the gradient oracle and the selected-inverse recurrence ------------------------------------------------------
@pytest.mark.parametrize("family", ["rbf", "vonkarman", "matern12", "matern32", "matern52"])
@pytest.mark.parametrize("ndim", [1, 2])
def test_oracle_gradient_against_central_differences(family, ndim):
    rng = np.random.default_rng(5 + ndim)
    n = 160
    X = rng.uniform(0, 6, size=(n, ndim))
    y = rng.normal(size=n)
    e2 = rng.uniform(0.01, 0.05, size=n)
    M = np.array([[1.3]]) if ndim == 1 else np.array([[1.1, 0.3], [0.3, 0.7]])
    amp = 1.7
    logl, g = gro.log_likelihood_gradient(family, X, y, e2, amp, M)
    ref, _ = go.log_likelihood(go.kmat(family, X, amp=amp, invLam=M) + np.diag(e2), y)
    assert logl == ref

    def ll(p):
        m = np.array([[p[1]]]) if ndim == 1 else np.array([[p[1], p[2]], [p[2], p[3]]])
        return go.log_likelihood(go.kmat(family, X, amp=np.exp(p[0]), invLam=m) + np.diag(e2), y)[0]

    p0 = np.array([np.log(amp), M[0, 0], 0.0 if ndim == 1 else M[0, 1], 0.0 if ndim == 1 else M[1, 1]])
    for j in range(2 if ndim == 1 else 4):
        e = np.zeros(4)
        e[j] = 1e-5
        fd = (ll(p0 + e) - ll(p0 - e)) / 2e-5
        assert abs(g[j] - fd) <= 1e-5 * max(1.0, np.max(np.abs(g))), (j, g[j], fd)
    if ndim == 1:
        assert g[2] == 0.0 and g[3] == 0.0


@pytest.mark.parametrize("field", [30.0, 4.0])
def test_selected_inverse_recurrence_on_the_envelope(field):
    """The recurrence tgp_selinv runs, restated in numpy on the envelope factor of gp_oracle.cholesky_envelope, equals
    np.linalg.inv on every envelope entry; Z[R, R] never leaves the envelope (asserted inside)."""
    rng = np.random.default_rng(9)
    n, block = 700, 64
    X = np.sort(rng.uniform(0, field, size=(n, 2)), axis=0)
    X[:, 1] = rng.uniform(0, field, size=n)
    X = X[np.argsort(X[:, 0], kind="stable")]
    K = go.kmat("rbf", X, amp=2.0, length_scale=0.35) + np.diag(rng.uniform(0.01, 0.02, size=n))
    dcut = 0.35 * np.sqrt(185.0)
    c1 = np.minimum(np.arange(block, n + block, block), n)
    row_end = np.maximum(np.searchsorted(X[:, 0], X[c1 - 1, 0] + dcut * (1 + 1e-9), side="left"), c1)
    L = go.cholesky_envelope(np.tril(K), row_end, block=block)
    Z, inside = gro.selected_inverse_envelope(L, row_end, block=block)
    ref = np.linalg.inv(K)
    assert np.all(np.isnan(Z[~inside])) and not np.any(np.isnan(Z[inside]))
    assert np.max(np.abs(Z[inside] - ref[inside])) <= 1e-10 * np.max(np.abs(ref))
    if field == 30.0:
        assert (~inside).any()   # a real envelope
    else:
        assert inside.all()      # the dense case is the same code


def test_new_entry_points_reject_bad_arguments_without_a_gpu():
    """Argument validation happens before any CUDA call."""
    from treegp_b200 import _cabi

    lib = _cabi.load()
    A16 = ctypes.c_void_p(16)
    re2 = np.array([1000, 1000], dtype=np.int64)
    rep = ctypes.c_void_p(re2.ctypes.data)
    assert lib.tgp_selinv_work_doubles(1000) >= 2 * 512 * 512 + 512 * 1000
    assert lib.tgp_selinv(None, 1000, 1000, None, 0, A16, None) == -1
    assert lib.tgp_selinv(A16, 1000, 1001, None, 0, A16, None) == -1                 # odd ld
    assert lib.tgp_selinv(A16, 1000, 1000, rep, 3, A16, None) == -1                  # 2 blocks, not 3
    assert b"row_end" in lib.tgp_last_error()
    assert lib.tgp_selinv(A16, 1000, 1000, rep, 2, None, None) == -1                 # no scratch
    assert b"scratch" in lib.tgp_last_error()
    ok = _cabi.TgpKernel(0, 2, 1.0, 1.0, 0.0, 1.0)
    bad = _cabi.TgpKernel(99, 2, 1.0, 1.0, 0.0, 1.0)
    args = [A16, A16, A16, 1000, ctypes.byref(ok), A16, 1000, A16, A16, A16, rep, 2, A16, None]
    for i, v in ((4, ctypes.byref(bad)), (0, None), (6, 999), (11, 1), (12, ctypes.c_void_p(8))):
        a = list(args)
        a[i] = v
        assert lib.tgp_loglike_grad(*a) == -1, i
