"""Test helper: numpy restatements for the analytic log-likelihood gradient and the selected inverse.

Not an algorithm of the reference, which fits with scipy's forward-difference gradient (log_likelihood.py:56-57): the
closed-form gradient it approximates, the profile derivatives f'(q), and the blocked Takahashi recurrence that
tgp_selinv runs.  Built on the pinned oracle (oracle/gp_oracle.py: kmat, log_likelihood) and checked against central
differences of it and against np.linalg.inv (tests/test_cpu_loglike_grad.py).
"""
import numpy as np
from scipy import special
from scipy.linalg import solve_triangular

from oracle.gp_oracle import kmat, log_likelihood


def profile_dq(family, q):
    """df/dq of the correlation profiles of kmat as functions of q = d^2 (q > 0): closed forms, and for the von Karman
    profile f = 2^(1/6)/Gamma(5/6) z^(5/6) K_{5/6}(z), z = 2 pi sqrt(q):  df/dq = -2 pi^2 2^(1/6)/Gamma(5/6)
    z^(-1/6) K_{1/6}(z)."""
    q = np.asarray(q, dtype=float)
    r = np.sqrt(q)
    if family == "rbf":
        return -0.5 * np.exp(-0.5 * q)
    if family == "matern12":
        return -0.5 * np.exp(-r) / r
    if family == "matern32":
        return -1.5 * np.exp(-np.sqrt(3.0) * r)
    if family == "matern52":
        s = np.sqrt(5.0) * r
        return -5.0 / 6.0 * (1.0 + s) * np.exp(-s)
    if family == "vonkarman":
        z = 2.0 * np.pi * r
        return -2.0 * np.pi ** 2 * 2.0 ** (1.0 / 6.0) / special.gamma(5.0 / 6.0) * z ** (-1.0 / 6.0) * special.kv(1.0 / 6.0, z)
    raise ValueError(family)


def log_likelihood_gradient(family, X, y, yerr2, amp, invLam):
    """log_likelihood of K = amp f(q) + diag(yerr2), q = delta^T invLam delta, and its gradient with respect to
    (ln amp, m00, m01, m11) -- dense K^-1 and explicit dK:  d logL / d t = 1/2 tr((alpha alpha^T - K^-1) dK/dt).
    1-D: invLam is 1 x 1 and the last two components are 0.  Not in the reference, which fits with a forward-difference
    gradient (log_likelihood.py:56-57); this is the standard closed form it approximates."""
    X = np.asarray(X, dtype=float)
    X = X[:, None] if X.ndim == 1 else X
    M = np.atleast_2d(np.asarray(invLam, dtype=float))
    K0 = kmat(family, X, amp=amp, invLam=M)
    logl, alpha = log_likelihood(K0 + np.diag(yerr2), y)
    Kinv = np.linalg.inv(K0 + np.diag(yerr2))
    W = np.outer(alpha, alpha) - Kinv
    dX = X[:, None, :] - X[None, :, :]
    q = np.einsum("pqi,ij,pqj->pq", dX, M, dX)
    fq = np.zeros_like(q)
    nz = q > 0
    fq[nz] = profile_dq(family, q[nz])
    dK = [K0]
    if X.shape[1] == 1:
        dK += [amp * fq * dX[:, :, 0] ** 2, np.zeros_like(q), np.zeros_like(q)]
    else:
        dK += [amp * fq * dX[:, :, 0] ** 2, amp * fq * 2.0 * dX[:, :, 0] * dX[:, :, 1], amp * fq * dX[:, :, 1] ** 2]
    return logl, np.array([0.5 * np.sum(W * d) for d in dK])


def selected_inverse_envelope(L, row_end, block=512):
    """Restatement (numpy, small cases) of tgp_selinv: Z = (L L^T)^-1 on the envelope of the factor L (as returned by
    cholesky_envelope with the same row_end / block) by the blocked Takahashi recurrence, block columns last to first:
        W = L11^-1,  T = L21 W,  Z[R, J] = -Z[R, R] T,  Z[J, J] = W^T W - T^T Z[R, J]
    with R = [end of J, row_end[J]).  Returns (Z, inside): Z holds NaN outside the envelope (never computed), `inside`
    is the boolean mask of the envelope (both triangles).  Raises if some Z[R, R] needed a value outside it."""
    L = np.asarray(L, dtype=float)
    n = L.shape[0]
    starts = list(range(0, n, block))
    re, prev = [], 0
    for b, k in enumerate(starts):
        c1 = min(n, k + block)
        prev = min(n, max(int(row_end[b]), prev, c1))
        re.append(prev)
    inside = np.zeros((n, n), dtype=bool)
    for b, k in enumerate(starts):
        c1 = min(n, k + block)
        inside[k:re[b], k:c1] = True
    inside |= inside.T
    Z = np.full((n, n), np.nan)
    for b in reversed(range(len(starts))):
        k = starts[b]
        c1 = min(n, k + block)
        R = slice(c1, re[b])
        W = solve_triangular(np.tril(L[k:c1, k:c1]), np.eye(c1 - k), lower=True)
        ZJJ = W.T @ W
        if re[b] > c1:
            if not inside[R, R].all():
                raise AssertionError("Z[R, R] leaves the envelope at block column %d" % b)
            T = L[R, k:c1] @ W
            ZRJ = -Z[R, R] @ T
            Z[R, k:c1], Z[k:c1, R] = ZRJ, ZRJ.T
            ZJJ = ZJJ - T.T @ ZRJ
        Z[k:c1, k:c1] = 0.5 * (ZJJ + ZJJ.T)
    return Z, inside
