"""Test helper: numpy oracle for sum kernels -- K = sum_c amp_c f_c(q_c) + white I (+ diag(y_err^2)), the reference's
generic `kernel(X) + eye * y_err**2` for a scikit-learn Sum of stationary terms and a WhiteKernel, and the closed-form
log-likelihood gradient with respect to (ln amp_c, m00_c, m01_c, m11_c) per term and ln white.

Built on the pinned oracle (oracle/gp_oracle.py: kmat, log_likelihood) and tests/grad_oracle.py (profile_dq) without
changing them.  A term is (family, amp, invLam) with the family names of gp_oracle.kmat.
"""
import numpy as np

from oracle.gp_oracle import kmat, log_likelihood
import grad_oracle as gro


def _coincident_off_diagonal(X):
    same = np.all(X[:, None, :] == X[None, :, :], axis=-1)
    np.fill_diagonal(same, False)
    return same


def term_kmat(term, X, Y=None):
    """amp f(q) of one term; in K(X, X) a von Karman term is 0 between distinct coincident points (the reference's
    pdist filter, kernels.py:253-262), an RBF / Matern term is not."""
    family, amp, M = term
    X = np.atleast_2d(np.asarray(X, dtype=float))
    K = kmat(family, X, Y, amp=amp, invLam=np.atleast_2d(M))
    if Y is None and family == "vonkarman":
        K[_coincident_off_diagonal(X)] = 0.0
    return K


def sum_kmat(terms, X, Y=None, white=0.0):
    """K(X, X) = sum of the terms + white I;  K(X, Y) = sum of the terms (sklearn's WhiteKernel(X, Y) is 0)."""
    K = sum(term_kmat(t, X, Y) for t in terms)
    if Y is None:
        K = K + white * np.eye(K.shape[0])
    return K


def sum_log_likelihood_gradient(terms, white, X, y, yerr2):
    """(logL, g) of K = sum_kmat(terms, X, white=white) + diag(yerr2); g = [d logL / d (ln amp_c, m00_c, m01_c, m11_c)
    for every term c..., d logL / d ln white] from d logL / d t = 1/2 tr((alpha alpha^T - K^-1) dK / dt).  1-D terms
    have zero m01 / m11 components."""
    X = np.asarray(X, dtype=float)
    X = X[:, None] if X.ndim == 1 else X
    K = sum_kmat(terms, X, white=white) + np.diag(yerr2)
    logl, alpha = log_likelihood(K, y)
    W = np.outer(alpha, alpha) - np.linalg.inv(K)
    dX = X[:, None, :] - X[None, :, :]
    g = []
    for family, amp, M in terms:
        M = np.atleast_2d(M)
        q = np.einsum("pqi,ij,pqj->pq", dX, M, dX)
        fq = np.zeros_like(q)
        nz = q > 0
        fq[nz] = gro.profile_dq(family, q[nz])
        dK = [term_kmat((family, amp, M), X)]
        if X.shape[1] == 1:
            dK += [amp * fq * dX[:, :, 0] ** 2, np.zeros_like(q), np.zeros_like(q)]
        else:
            dK += [amp * fq * dX[:, :, 0] ** 2, amp * fq * 2.0 * dX[:, :, 0] * dX[:, :, 1], amp * fq * dX[:, :, 1] ** 2]
        g += [0.5 * np.sum(W * d) for d in dK]
    g.append(0.5 * white * np.trace(W))
    return logl, np.array(g)


def terms_of(desc):
    """(terms, white) of a TgpKernelSum, for the functions above."""
    names = {0: "rbf", 1: "vonkarman", 2: "matern12", 3: "matern32", 4: "matern52"}
    terms = []
    for c in range(desc.nterms):
        t = desc.term[c]
        M = np.array([[t.m00]]) if desc.ndim == 1 else np.array([[t.m00, t.m01], [t.m01, t.m11]])
        terms.append((names[t.family], t.amp, M))
    return terms, desc.white
