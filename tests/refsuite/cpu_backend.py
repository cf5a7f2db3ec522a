"""TEST INFRASTRUCTURE: a CPU stand-in for treegp_b200.backend built on the oracle.

Used only by tests/golden_r2_checks.py to run the host logic around the device operators (optimiser loops,
bootstrap bookkeeping, E/B utilities) on a machine without a GPU; it does not check the CUDA arithmetic -- that
is what the `-m gpu` parity tests are for.  The product never imports this module.
"""
import numpy as np
import scipy.linalg as sla
import torch

from oracle import gp_oracle as go
from oracle import pairbin_oracle as po
from treegp_b200 import _cabi, backend

_FAM = {_cabi.FAM_RBF: "rbf", _cabi.FAM_VONKARMAN: "vonkarman", _cabi.FAM_MATERN12: "matern12",
        _cabi.FAM_MATERN32: "matern32", _cabi.FAM_MATERN52: "matern52"}
F64 = torch.float64


def _np(t):
    return t.numpy() if isinstance(t, torch.Tensor) else np.asarray(t)


def _metric(d):
    return np.array([[d.m00]]) if d.ndim == 1 else np.array([[d.m00, d.m01], [d.m01, d.m11]])


def _kmat(d, X, Y=None):
    X = _np(X)
    K = go.kmat(_FAM[d.family], X, None if Y is None else _np(Y), amp=d.amp, invLam=_metric(d))
    if Y is None and d.family == _cabi.FAM_VONKARMAN:  # reference quirk, kernels.py:253-262
        same = (np.abs(X[:, None, :] - X[None, :, :]).sum(-1) == 0) & ~np.eye(len(X), dtype=bool)
        K[same] = 0.0
    return K


def install():
    dev = torch.device("cpu")
    backend.require_cuda = lambda: dev

    def to_device(a, dtype=F64, non_blocking=False):
        if isinstance(a, torch.Tensor):
            return a.to(dtype=dtype).contiguous()
        return torch.as_tensor(np.ascontiguousarray(a), dtype=dtype)

    backend.to_device = to_device

    def kmat_sym(X, kdesc, diag_add=None, out=None, lower_only=False):
        X = backend.as_points(X)
        n = X.shape[0]
        out = backend.alloc_matrix(n, n) if out is None else out
        K = _kmat(kdesc, X)
        if diag_add is not None:
            K = K + np.diag(_np(diag_add))
        out[:n, :n] = torch.as_tensor(K)
        return out

    def kmat_cross(Xs, X, kdesc, out=None):
        Xs, X = backend.as_points(Xs), backend.as_points(X)
        out = backend.alloc_matrix(Xs.shape[0], X.shape[0]) if out is None else out
        out[:Xs.shape[0], :X.shape[0]] = torch.as_tensor(_kmat(kdesc, Xs, X))
        return out

    def potrf(A, N, row_end=None):
        info = torch.zeros(1, dtype=torch.int32)
        K = np.tril(_np(A[:N, :N]))
        K = K + np.tril(K, -1).T
        try:
            L = sla.cholesky(K, lower=True)
        except np.linalg.LinAlgError as e:
            import re
            m = re.match(r"(\d+)", str(e))
            info[0] = int(m.group(1)) if m else 1
            return info
        il = np.tril_indices(N)
        An = _np(A)
        An[:N, :N][il] = L[il]
        return info

    def potrs_vec(L, N, b):
        b[:] = torch.as_tensor(sla.cho_solve((np.tril(_np(L[:N, :N])), True), _np(b)))
        return b

    def trsm_rows(L, N, B, M, row_end=None):
        B[:M, :N] = torch.as_tensor(sla.solve_triangular(np.tril(_np(L[:N, :N])), _np(B[:M, :N]).T, lower=True).T)
        return B

    def gemm_nt_sub(C, M, Nc, A, B, Kd, lower_only=False):
        upd = _np(A[:M, :Kd]) @ _np(B[:Nc, :Kd]).T
        if lower_only:
            upd = np.tril(upd)
        C[:M, :Nc] -= torch.as_tensor(upd)
        return C

    def loglike(X, y, yerr2, kdesc, work=None, want_alpha=False, row_end=None):
        X = backend.as_points(X)
        n = X.shape[0]
        Y = _np(y)
        cols = [Y] if Y.ndim == 1 else [Y[:, c] for c in range(Y.shape[1])]   # y (n,) or (n, r): the joint logL
        work = backend.alloc_matrix(n + len(cols), n) if work is None else work
        K = _kmat(kdesc, X) + np.diag(_np(yerr2))
        fits = [go.log_likelihood(K, c) for c in cols]
        info = torch.zeros(1, dtype=torch.int32)
        out = torch.zeros(3, dtype=F64)
        if fits[0][1] is None:
            info[0] = 1
            out[0] = -np.inf
            alpha = np.zeros(Y.shape)
        else:
            out[0] = sum(logl for logl, _ in fits)
            alpha = fits[0][1] if Y.ndim == 1 else np.stack([a for _, a in fits], axis=1)
            il = np.tril_indices(n)
            _np(work)[:n, :n][il] = sla.cholesky(K, lower=True)[il]   # the factor stays in the workspace
        return out, info, torch.as_tensor(alpha), work

    def predict_mean(Xs, X, kdesc, alpha, out=None):
        return torch.as_tensor(_kmat(kdesc, backend.as_points(Xs), backend.as_points(X)) @ _np(alpha))

    def predict_var(Xs, X, kdesc, L, chunk=None, out=None, work=None, row_end=None):
        Ks = _kmat(kdesc, backend.as_points(Xs), backend.as_points(X))
        n = Ks.shape[1]
        V = sla.solve_triangular(np.tril(_np(L[:n, :n])), Ks.T, lower=True)
        return torch.as_tensor(kdesc.amp - np.sum(V * V, axis=0))

    def pairbin(px, py, pk, pw, cat_off, max_cat_len, bin_type, edges, nbins, min_sep, max_sep, rank=0, nranks=1):
        bt = "TwoD" if bin_type == _cabi.BIN_TWOD else "Log"
        off = _np(cat_off)
        rows = []
        for c in range(len(off) - 1):
            s = slice(int(off[c]), int(off[c + 1]))
            if off[c + 1] - off[c] < 2:
                nb = nbins * nbins if bt == "TwoD" else nbins
                r = dict(npairs=np.zeros(nb, np.int64), weight=np.zeros(nb), sumwkk=np.zeros(nb), sumwr=np.zeros(nb))
            else:
                r = po.pairbin(_np(px[s]), _np(py[s]), _np(pk[s]), None if pw is None else _np(pw[s]), min_sep, max_sep,
                               nbins, bt)
            rows.append(r)
        st = lambda key: torch.as_tensor(np.stack([r[key] for r in rows]))
        return st("npairs"), st("weight"), st("sumwkk"), (st("sumwr") if bt == "Log" else None)

    def pairbin_packed(px, py, pk, pw, cat_off, max_cat_len, bin_type, edges, nbins, min_sep, max_sep, rank=0, nranks=1):
        npairs, sw, swkk, swr = pairbin(px, py, pk, pw, cat_off, max_cat_len, bin_type, edges, nbins, min_sep, max_sep)
        planes = [npairs.to(torch.int64).view(F64), sw, swkk] + ([] if swr is None else [swr])
        return torch.stack(planes)

    backend.pairbin_packed = pairbin_packed
    from . import bootbin_standin

    bootbin_standin.install(backend, po)

    def robust_chi2_batch(coord_d, y_d, W_d, family, params):
        """numpy restatement of two_pcf.py:12-31,96-148 (the objective of the robust fit) for the stand-in."""
        coord, yv, W = _np(coord_d), _np(y_d), _np(W_d)
        out = np.zeros((len(params), 4))
        for i, (size, g1, g2) in enumerate(np.asarray(params, dtype=float).reshape(-1, 3)):
            if not np.isfinite(size + g1 + g2) or abs(g1) > 1 or abs(g2) > 1:
                out[i, 0] = np.inf
                continue
            e = np.sqrt(g1 ** 2 + g2 ** 2)
            q = (1 - e) / (1 + e)
            phi = 0.5 * np.arctan2(g2, g1)
            rot = np.array([[np.cos(phi), np.sin(phi)], [-np.sin(phi), np.cos(phi)]])
            Lm = rot.T @ np.diag([size ** 2, (size * q) ** 2]) @ rot
            model = go.kmat(_FAM[family], coord, np.zeros((1, 2)), amp=1.0, invLam=np.linalg.inv(Lm))[:, 0]
            F = np.array([model, np.ones_like(model)]).T
            FtW = F.T @ W
            alpha = np.linalg.inv(FtW @ F) @ (FtW @ yv)
            alpha[0] = abs(alpha[0])
            r = yv - (alpha[0] * model + alpha[1])
            out[i] = [r @ W @ r, alpha[0], alpha[1], 1.0]
        return out

    backend.robust_chi2_batch = robust_chi2_batch

    def knn_mean(X0, y0, Xq, k):
        from sklearn.neighbors import KNeighborsRegressor   # what the reference itself calls (gp_interp.py:236-238)

        return torch.as_tensor(KNeighborsRegressor(n_neighbors=k).fit(_np(X0), _np(y0)).predict(_np(Xq)))

    backend.knn_mean = knn_mean

    def vcorr_sums(x, y, dx, dy, logrmin, dlogr, bins):
        from oracle import eb_oracle

        return eb_oracle.pair_sums(*(np.asarray(a, dtype=float) for a in (x, y, dx, dy)), logrmin, dlogr, bins)

    backend.vcorr_sums = vcorr_sums
    backend.kmat_sym, backend.kmat_cross, backend.potrf, backend.potrs_vec = kmat_sym, kmat_cross, potrf, potrs_vec
    backend.trsm_rows, backend.gemm_nt_sub, backend.loglike = trsm_rows, gemm_nt_sub, loglike
    backend.predict_mean, backend.predict_var, backend.pairbin = predict_mean, predict_var, pairbin
    # the dense stand-ins above are what the host logic is checked against: no envelopes, no variance windows
    backend.plan_envelope = lambda *a, **k: None
    backend.predict_var_windowed = lambda *a, **k: None
    backend.hilbert_order = lambda px, py: torch.arange(px.numel())
