"""Test helper: numpy oracle for several outputs sharing one kernel -- r independent GPs with the covariance
K = sum_kmat(terms, X, white) + diag(y_err^2): the joint log-likelihood sum_c logL_c (scikit-learn's
GaussianProcessRegressor.log_marginal_likelihood for multi-target y) and its closed-form gradient
    d logL / d t = 1/2 tr((A A^T - r K^-1) dK / dt),  A = K^-1 Y,
with respect to (ln amp_c, m00_c, m01_c, m11_c) per term and ln white, in the layout of
sum_oracle.sum_log_likelihood_gradient.  Built on tests/sum_oracle.py and tests/grad_oracle.py without changing them.
"""
import numpy as np

import grad_oracle as gro
import sum_oracle as so


def _dK(terms, white, X):
    """dK / d (ln amp_c, m00_c, m01_c, m11_c) for every term, then dK / d ln white."""
    dX = X[:, None, :] - X[None, :, :]
    out = []
    for family, amp, M in terms:
        M = np.atleast_2d(M)
        q = np.einsum("pqi,ij,pqj->pq", dX, M, dX)
        fq = np.zeros_like(q)
        nz = q > 0
        fq[nz] = gro.profile_dq(family, q[nz])
        out.append(so.term_kmat((family, amp, M), X))
        if X.shape[1] == 1:
            out += [amp * fq * dX[:, :, 0] ** 2, np.zeros_like(q), np.zeros_like(q)]
        else:
            out += [amp * fq * dX[:, :, 0] ** 2, amp * fq * 2.0 * dX[:, :, 0] * dX[:, :, 1], amp * fq * dX[:, :, 1] ** 2]
    out.append(white * np.eye(X.shape[0]))
    return out


def joint_log_likelihood_gradient(terms, white, X, Y, yerr2):
    """(joint logL, g, A): logL = -1/2 sum_c y_c^T K^-1 y_c - r/2 ln|K| - r N/2 ln 2 pi, its gradient g and
    A = K^-1 Y (N, r)."""
    X = np.asarray(X, dtype=float)
    X = X[:, None] if X.ndim == 1 else X
    Y = np.asarray(Y, dtype=float)
    n, r = Y.shape
    K = so.sum_kmat(terms, X, white=white) + np.diag(yerr2)
    L = np.linalg.cholesky(K)
    A = np.linalg.solve(K, Y)
    logl = -0.5 * np.sum(Y * A) - r * np.sum(np.log(np.diag(L))) - 0.5 * r * n * np.log(2.0 * np.pi)
    W = A @ A.T - r * np.linalg.inv(K)
    g = np.array([0.5 * np.sum(W * d) for d in _dK(terms, white, X)])
    return logl, g, A
