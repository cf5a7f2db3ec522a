"""GPU: predictive variance and leave-one-out predictions of a batch (tgp_predict_var_batch, tgp_loo_batch) -- bit for
bit against tgp_predict_var_sum / GPInterpolation.loo_predict on each problem alone, against an independent scipy
oracle and explicit refits, independence of the problems and of both chunkings, and GPInterpolationBatch.predict_var /
loo_predict against per-problem GPInterpolation, including the errors they raise."""
import ctypes

import numpy as np
import pytest
import torch
from scipy import linalg

from test_gpu_batch import KERNELS_1D, KERNELS_2D, SIZES, _problems, _single

pytestmark = pytest.mark.gpu

MS = [0, 1, 63, 64, 65, 1000]


def _test_points(probs, ms, seed):
    from treegp_b200 import backend

    rng = np.random.default_rng(seed)
    out = []
    for p, m in zip(probs, ms):
        n, ndim = p[0].shape
        side = max(n, 1) ** (1.0 / ndim) * 1.5
        out.append(backend.to_device(rng.uniform(-1, side + 1, size=(m, ndim))))
    return out


def _var_batch(probs, xs, budget=4 << 30):
    from treegp_b200 import backend

    X, y, e2 = (torch.cat([p[k] for p in probs]) for k in range(3))
    return backend.predict_var_batch(torch.cat(xs), [x.shape[0] for x in xs], X, y, e2, [p[0].shape[0] for p in probs],
                                     [p[3] for p in probs], budget_bytes=budget)


def _var_raw(probs, xs, chunk):
    """One call of the C entry on the factors of one tgp_loglike_batch call, with the given chunk."""
    from treegp_b200 import _cabi, backend

    sizes, ssizes = [p[0].shape[0] for p in probs], [x.shape[0] for x in xs]
    off, soff = backend.batch_offsets(sizes), backend.batch_offsets(ssizes)
    dev = probs[0][0].device
    X, y, e2 = (torch.cat([p[k] for p in probs]) for k in range(3))
    work = torch.empty(backend.batch_work_doubles(sizes), dtype=torch.float64, device=dev)
    out = torch.empty((len(probs), 3), dtype=torch.float64, device=dev)
    info = torch.empty(len(probs), dtype=torch.int32, device=dev)
    alpha = torch.empty(int(off[-1]), dtype=torch.float64, device=dev)
    ks = backend._ksum_array([p[3] for p in probs])
    lib = _cabi.load()
    _cabi.check(lib.tgp_loglike_batch(backend._p(X), backend._p(y), backend._p(e2), backend._host_i64(off), len(probs),
                                      ctypes.cast(ks, ctypes.c_void_p), backend._p(work), backend._p(alpha), 0,
                                      backend._p(out), backend._p(info), backend._stream()))
    vwork = torch.empty(int(lib.tgp_predict_var_batch_work_doubles(backend._host_i64(soff), backend._host_i64(off),
                                                                   len(probs), chunk)),
                        dtype=torch.float64, device=dev)
    var = torch.full((int(soff[-1]),), float("nan"), dtype=torch.float64, device=dev)
    Xs = torch.cat(xs)
    _cabi.check(lib.tgp_predict_var_batch(backend._p(Xs), backend._host_i64(soff), backend._p(X), backend._host_i64(off),
                                          len(probs), ctypes.cast(ks, ctypes.c_void_p), backend._p(work),
                                          backend._p(vwork), chunk, backend._p(var), backend._stream()),
                "tgp_predict_var_batch")
    assert torch.all(info == 0)
    return var


def _var_single(p, x, chunk=None):
    """tgp_predict_var_sum (dense) on the factor of tgp_loglike_sum for one problem."""
    from treegp_b200 import backend

    _, info, _, work = _single(p)
    assert int(info.item()) == 0
    if x.shape[0] == 0:
        return torch.empty(0, dtype=torch.float64, device=x.device)
    return backend.predict_var(x, p[0], backend.as_sum(p[3]), work, chunk=chunk)


def _split(t, sizes):
    return list(torch.split(t, [int(s) for s in sizes]))


@pytest.mark.parametrize("ndim,kstrs", [(2, KERNELS_2D), (1, KERNELS_1D)], ids=["2d", "1d"])
def test_var_batch_bitwise_against_single(gpu_ready, ndim, kstrs):
    # every size with two test-point counts and every kernel (the sizes run through both lists at different strides)
    probs = _problems(SIZES, ndim, kstrs, seed=60 + ndim) + _problems(SIZES, ndim, kstrs[2:] + kstrs[:2], seed=70)
    ms = [MS[b % len(MS)] for b in range(len(SIZES))] + [MS[(b + 3) % len(MS)] for b in range(len(SIZES))]
    xs = _test_points(probs, ms, seed=80 + ndim)
    var, info = _var_batch(probs, xs)
    assert torch.all(info == 0)
    for b, v in enumerate(_split(var, ms)):
        assert torch.equal(v, _var_single(probs[b], xs[b])), (b, probs[b][0].shape[0], ms[b])
    # the raw entry with the largest chunk it accepts gives the same rows
    assert torch.equal(_var_raw(probs, xs, 1000), var)


def test_var_batch_against_cho_solve_oracle(gpu_ready):
    from treegp_b200 import eval_kernel

    kstrs = [KERNELS_2D[0], KERNELS_2D[3], KERNELS_2D[6]]
    probs = _problems([40, 90, 130], 2, kstrs, seed=5)
    xs = _test_points(probs, [30, 50, 20], seed=6)
    var, info = _var_batch(probs, xs)
    assert torch.all(info == 0)
    for b, v in enumerate(_split(var, [30, 50, 20])):
        X, e2 = probs[b][0].cpu().numpy(), probs[b][2].cpu().numpy()
        Xs = xs[b].cpu().numpy()
        k = eval_kernel(kstrs[b])
        K = k.__call__(X) + np.diag(e2)
        Ks = k.__call__(Xs, X)
        prior = float(np.max(np.diag(k.__call__(Xs))))   # k(0): the white level is on the diagonal of K(Xs, Xs)
        ref = prior - np.sum(Ks * linalg.cho_solve(linalg.cho_factor(K, lower=True), Ks.T).T, axis=1)
        assert np.max(np.abs(v.cpu().numpy() - ref)) <= 1e-10 * prior, b


def test_var_batch_independent_of_order_subsets_chunking_and_repeats(gpu_ready):
    from treegp_b200 import backend

    sizes = [700, 65, 1536, 1, 2000, 300]
    ms = [257, 64, 90, 3, 130, 0]
    probs = _problems(sizes, 2, KERNELS_2D, seed=21)
    xs = _test_points(probs, ms, seed=22)
    ref, _ = _var_batch(probs, xs)
    refs = _split(ref, ms)
    perm = [4, 2, 0, 5, 3, 1]
    v, _ = _var_batch([probs[i] for i in perm], [xs[i] for i in perm])
    for j, i in enumerate(perm):
        assert torch.equal(_split(v, [ms[i] for i in perm])[j], refs[i])
    v, _ = _var_batch([probs[i] for i in (1, 4)], [xs[i] for i in (1, 4)])
    assert torch.equal(v, torch.cat([refs[1], refs[4]]))
    # a budget just above the largest factor: three chunks of problems, and 7 test points per pass for N = 2000
    budget = 8 * backend.batch_work_doubles([2000]) + 8 * 2000 * 7
    assert backend.plan_batch_chunks(sizes, budget) == [(0, 4), (4, 5), (5, 6)]
    assert backend.var_batch_chunk([130], [2000], budget) == 7
    v, _ = _var_batch(probs, xs, budget=budget)
    assert torch.equal(v, ref)
    assert torch.equal(_var_raw(probs, xs, 1), ref)
    assert torch.equal(_var_raw(probs, xs, 65), ref)
    v, _ = _var_batch(probs, xs)
    assert torch.equal(v, ref)


def _loo_batch(probs):
    from treegp_b200 import backend

    X, y, e2 = (torch.cat([p[k] for p in probs]) for k in range(3))
    return backend.loo_batch(X, y, e2, [p[0].shape[0] for p in probs], [p[3] for p in probs])


def _gp(p, kstr, monkeypatch):
    import treegp_b200 as treegp

    monkeypatch.setattr(treegp.GPInterpolation, "BANDED_SOLVE", False)
    monkeypatch.setattr(treegp.GPInterpolation, "WINDOWED_VARIANCE", False)
    gp = treegp.GPInterpolation(kernel=kstr, optimizer="none", normalize=False)
    gp.initialize(p[0].cpu().numpy(), p[1].cpu().numpy(), y_err=np.sqrt(p[2].cpu().numpy()))
    return gp


@pytest.mark.parametrize("ndim,kstrs", [(2, KERNELS_2D), (1, KERNELS_1D)], ids=["2d", "1d"])
def test_loo_batch_against_single_loo_predict(gpu_ready, monkeypatch, ndim, kstrs):
    from treegp_b200 import backend

    sizes = [1, 2, 63, 65, 512, 513, 1536, 2000]
    # errors whose square is what GPInterpolation squares on the host, so that both paths add the same yerr2
    probs = [(X, y, backend.to_device(np.sqrt(e2.cpu().numpy()) ** 2), d)
             for X, y, e2, d in _problems(sizes, ndim, kstrs, seed=90 + ndim)]
    mean, var, info = _loo_batch(probs)
    assert torch.all(info == 0)
    for b, (m, v) in enumerate(zip(_split(mean, sizes), _split(var, sizes))):
        m1, v1 = _gp(probs[b], kstrs[b % len(kstrs)], monkeypatch).loo_predict()
        assert np.array_equal(v.cpu().numpy(), v1), (b, sizes[b])
        assert np.max(np.abs(m.cpu().numpy() - m1)) <= 1e-9 * np.max(np.abs(m1)), (b, sizes[b])


def test_loo_batch_bitwise_var_and_refits(gpu_ready, monkeypatch):
    import treegp_b200 as treegp

    # errors given as exact squares on the host, so that the single path's y_err ** 2 is the batch's yerr2
    rng = np.random.default_rng(11)
    kstr = "1.5 * AnisotropicRBF(invLam=array([[0.5, 0.1], [0.1, 0.8]]))"
    n = 40
    X = rng.uniform(0, 9, size=(n, 2))
    y = rng.normal(size=n)
    yerr = rng.uniform(0.05, 0.1, size=n)
    gb = treegp.GPInterpolationBatch(kernel=kstr, optimizer="none", normalize=False)
    gb.initialize([X, X[:17]], [y, y[:17]], [yerr, yerr[:17]])
    means, vars_ = gb.loo_predict()
    monkeypatch.setattr(treegp.GPInterpolation, "BANDED_SOLVE", False)
    for Xb, yb, eb, mb, vb in [(X, y, yerr, means[0], vars_[0]), (X[:17], y[:17], yerr[:17], means[1], vars_[1])]:
        gp = treegp.GPInterpolation(kernel=kstr, optimizer="none", normalize=False)
        gp.initialize(Xb, yb, y_err=eb)
        m1, v1 = gp.loo_predict()
        assert np.array_equal(vb, v1)
        assert np.max(np.abs(mb - m1)) <= 1e-9 * np.max(np.abs(m1))
    for i in range(0, n, 7):   # explicit refits without point i
        keep = np.arange(n) != i
        gp = treegp.GPInterpolation(kernel=kstr, optimizer="none", normalize=False)
        gp.initialize(X[keep], y[keep], y_err=yerr[keep])
        mi, vi = gp.predict_var(X[i:i + 1])
        assert abs(means[0][i] - mi[0]) <= 1e-8 * max(1.0, abs(mi[0])), i
        assert abs(vars_[0][i] - vi[0]) <= 1e-8, i


def test_gp_batch_predict_var_and_loo_against_gpinterpolation(gpu_ready, monkeypatch):
    import treegp_b200 as treegp

    monkeypatch.setattr(treegp.GPInterpolation, "BANDED_SOLVE", False)
    monkeypatch.setattr(treegp.GPInterpolation, "WINDOWED_VARIANCE", False)
    rng = np.random.default_rng(31)
    sizes = [120, 700, 1, 1300]
    kstrs = ["2.0 * AnisotropicVonKarman(invLam=array([[0.9, -0.35], [-0.35, 0.6]]))",
             "ConstantKernel(1.1) * Matern(0.8, nu=1.5)", "ConstantKernel(1.3) * RBF(1.2)",
             "ConstantKernel(1.2) * RBF(0.9) + 0.4 * Matern(2.0, nu=1.5) + WhiteKernel(0.03)"]
    Xs = [rng.uniform(0, 1.5 * np.sqrt(n), size=(n, 2)) for n in sizes]
    ys = [rng.normal(size=n) + 3.0 for n in sizes]
    es = [rng.uniform(0.05, 0.1, size=n) for n in sizes]
    news = [rng.uniform(0, 1.5 * np.sqrt(n), size=(m, 2)) for n, m in zip(sizes, [50, 0, 7, 300])]
    gb = treegp.GPInterpolationBatch(kernel=kstrs, optimizer="none", normalize=True, white_noise=0.02)
    gb.initialize(Xs, ys, es)
    means, vars_ = gb.predict_var(news)
    pm = gb.predict(news)
    lm, lv = gb.loo_predict()
    for b in range(len(sizes)):
        gp = treegp.GPInterpolation(kernel=kstrs[b], optimizer="none", normalize=True, white_noise=0.02)
        gp.initialize(Xs[b], ys[b], y_err=es[b])
        assert np.array_equal(means[b], pm[b])
        if len(news[b]) == 0:
            assert vars_[b].shape == (0,)
            continue
        m1, v1 = gp.predict_var(news[b])
        assert np.array_equal(vars_[b], v1), b
        assert np.max(np.abs(means[b] - m1)) <= 1e-9 * max(1.0, np.max(np.abs(m1))), b
    for b in range(len(sizes)):
        gp = treegp.GPInterpolation(kernel=kstrs[b], optimizer="none", normalize=True, white_noise=0.02)
        gp.initialize(Xs[b], ys[b], y_err=es[b])
        lm1, lv1 = gp.loo_predict()
        assert np.array_equal(lv[b], lv1), b
        assert np.max(np.abs(lm[b] - lm1)) <= 1e-9 * np.max(np.abs(lm1)), b


def test_gp_batch_predict_var_and_loo_errors(gpu_ready):
    import treegp_b200 as treegp

    rng = np.random.default_rng(41)
    Xs = [rng.uniform(0, 10, size=(n, 2)) for n in (50, 40, 30)]
    ys = [rng.normal(size=n) for n in (50, 40, 30)]
    es = [np.full(n, 0.1) for n in (50, 40, 30)]
    es[1][10] = np.nan   # a NaN error: the pivot is not finite, so K_1 is not positive definite
    gb = treegp.GPInterpolationBatch(kernel="ConstantKernel(1.0) * RBF(3.0)", optimizer="none")
    gb.initialize(Xs, ys, es)
    with pytest.raises(np.linalg.LinAlgError, match="problem 1: .*not positive definite"):
        gb.predict_var([x[:3] for x in Xs])
    with pytest.raises(np.linalg.LinAlgError, match="problem 1: .*not positive definite"):
        gb.loo_predict()
    es[1][10] = 0.1
    gb.initialize(Xs, ys, es)
    gb.kernels[2] = gb.kernels[2].clone_with_theta(np.array([np.nan, 0.0]))
    with pytest.raises(np.linalg.LinAlgError, match="problem 2: the kernel has non-finite"):
        gb.predict_var([x[:3] for x in Xs])
    with pytest.raises(np.linalg.LinAlgError, match="problem 2: the kernel has non-finite"):
        gb.loo_predict()
