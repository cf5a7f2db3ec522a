"""GPU: batches of independent problems -- tgp_loglike_batch against tgp_loglike on each problem alone (bit for bit
without alpha, to 1e-10 with it), the batched mean against the untruncated single mean, independence of the
problems, chunking and repeatability, and GPInterpolationBatch against per-problem GPInterpolation runs."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

SIZES = [1, 2, 63, 64, 65, 511, 512, 513, 1535, 1536, 2000, 4096]
KERNELS_2D = ["2.0 * AnisotropicVonKarman(invLam=array([[0.9, -0.35], [-0.35, 0.6]]))",
              "1.5 * AnisotropicRBF(invLam=array([[0.5, 0.1], [0.1, 0.8]]))",
              "ConstantKernel(1.3) * RBF(1.2)",
              "ConstantKernel(0.9) * Matern(1.1, nu=0.5)",
              "ConstantKernel(1.1) * Matern(0.8, nu=1.5)",
              "ConstantKernel(0.7) * Matern(1.4, nu=2.5)",
              "ConstantKernel(1.2) * RBF(0.9) + 0.4 * Matern(2.0, nu=1.5) + WhiteKernel(0.03)"]
KERNELS_1D = ["2.0 * VonKarman(1.3)", "ConstantKernel(1.3) * RBF(1.2)", "ConstantKernel(0.9) * Matern(1.1, nu=0.5)",
              "ConstantKernel(1.1) * Matern(0.8, nu=1.5)", "ConstantKernel(0.7) * Matern(1.4, nu=2.5)",
              "ConstantKernel(1.2) * RBF(0.9) + 0.4 * Matern(2.0, nu=1.5) + WhiteKernel(0.03)"]


def _desc(kstr, ndim):
    from treegp_b200 import eval_kernel
    from treegp_b200.kernels import lower

    return lower(eval_kernel(kstr), ndim)


def _problems(sizes, ndim, kstrs, seed):
    """Points with density ~1 per unit area / length (well-conditioned K), values, errors, and a kernel per problem."""
    from treegp_b200 import backend

    rng = np.random.default_rng(seed)
    probs = []
    for b, n in enumerate(sizes):
        side = max(n, 1) ** (1.0 / ndim) * 1.5
        X = rng.uniform(0, side, size=(n, ndim))
        if n > 8:
            X[5] = X[2]                      # coincident points (the von Karman rule of K(X, X))
        probs.append((backend.to_device(X), backend.to_device(rng.normal(size=n)),
                      backend.to_device(rng.uniform(0.05, 0.1, size=n) ** 2), _desc(kstrs[b % len(kstrs)], ndim)))
    return probs


def _batch(probs, want_alpha=False, budget=4 << 30):
    from treegp_b200 import backend

    X = torch.cat([p[0] for p in probs])
    y = torch.cat([p[1] for p in probs])
    e2 = torch.cat([p[2] for p in probs])
    return backend.loglike_batch(X, y, e2, [p[0].shape[0] for p in probs], [p[3] for p in probs],
                                 want_alpha=want_alpha, budget_bytes=budget)


def _single(p, want_alpha=False):
    from treegp_b200 import backend

    return backend.loglike(p[0], p[1], p[2], p[3], want_alpha=want_alpha)


def _factor_block(work_single, n):
    return torch.tril(work_single[:n, :n])


@pytest.mark.parametrize("ndim,kstrs", [(2, KERNELS_2D), (1, KERNELS_1D)], ids=["2d", "1d"])
def test_loglike_batch_bitwise_against_single(gpu_ready, ndim, kstrs):
    from treegp_b200 import _cabi, backend

    probs = _problems(SIZES, ndim, kstrs, seed=10 + ndim)
    out, info, alpha = _batch(probs)
    # the factor blocks: one chunk, the workspace of the call itself
    sizes = [p[0].shape[0] for p in probs]
    off = backend.batch_offsets(sizes)
    work = torch.empty(backend.batch_work_doubles(sizes), dtype=torch.float64, device=gpu_ready)
    o2 = torch.empty((len(probs), 3), dtype=torch.float64, device=gpu_ready)
    i2 = torch.empty(len(probs), dtype=torch.int32, device=gpu_ready)
    a2 = torch.empty(int(off[-1]), dtype=torch.float64, device=gpu_ready)
    ks = backend._ksum_array([p[3] for p in probs])
    X, y, e2 = (torch.cat([p[k] for p in probs]) for k in range(3))
    import ctypes
    _cabi.check(_cabi.load().tgp_loglike_batch(backend._p(X), backend._p(y), backend._p(e2), backend._host_i64(off),
                                               len(probs), ctypes.cast(ks, ctypes.c_void_p), backend._p(work),
                                               backend._p(a2), 0, backend._p(o2), backend._p(i2), backend._stream()))
    assert torch.equal(o2, out) and torch.equal(i2, info) and torch.equal(a2, alpha)
    woff = 0
    for b, p in enumerate(probs):
        n = sizes[b]
        ld = (n + 1) // 2 * 2
        o1, i1, a1, w1 = _single(p)
        assert int(info[b]) == 0 and int(i1.item()) == 0
        assert torch.equal(out[b], o1), (b, n, out[b], o1)
        assert torch.equal(alpha[off[b]:off[b + 1]], a1), (b, n)
        blk = work[woff:woff + (n + 1) * ld].view(n + 1, ld)
        assert torch.equal(torch.tril(blk[:n, :n]), _factor_block(w1, n)), (b, n)
        woff += (n + 1) * ld
    # want_alpha: info and logdet bitwise, logL to 1e-12, alpha to 1e-10 of its largest entry
    outa, infoa, alphaa = _batch(probs, want_alpha=True)
    assert torch.equal(infoa, info)
    for b, p in enumerate(probs):
        o1, _, a1, _ = _single(p, want_alpha=True)
        assert float(outa[b, 2]) == float(o1[2])
        assert abs(float(outa[b, 0]) - float(o1[0])) <= 1e-12 * abs(float(o1[0])) + 1e-300
        ab = alphaa[off[b]:off[b + 1]]
        assert float((ab - a1).abs().max()) <= 1e-10 * float(a1.abs().max()), (b, sizes[b])


def test_predict_mean_batch_equals_single(gpu_ready):
    from treegp_b200 import backend

    sizes = [1, 63, 300, 1024, 700, 2000]
    kstrs = KERNELS_2D
    probs = _problems(sizes, 2, kstrs, seed=3)
    _, _, alpha = _batch(probs, want_alpha=True)
    off = backend.batch_offsets(sizes)
    rng = np.random.default_rng(4)
    ssizes = [5, 0, 257, 40, 1, 600]
    Xs = [backend.to_device(rng.uniform(0, 40, size=(m, 2))) for m in ssizes]
    mean = backend.predict_mean_batch(torch.cat(Xs), ssizes, torch.cat([p[0] for p in probs]), sizes,
                                      [p[3] for p in probs], alpha)
    soff = backend.batch_offsets(ssizes)
    for b, p in enumerate(probs):
        if ssizes[b] == 0:
            continue
        ref = backend.predict_mean(Xs[b], p[0], p[3], alpha[off[b]:off[b + 1]].contiguous(), truncate=False)
        got = mean[soff[b]:soff[b + 1]]
        if sizes[b] <= 1024:   # the single call sums in one pass: the same sum bit for bit
            assert torch.equal(got, ref), b
        else:                  # the single call splits the training tiles over CTAs (atomic partial sums)
            assert float((got - ref).abs().max()) <= 1e-12 * float(ref.abs().max())


def test_problems_are_independent(gpu_ready):
    sizes = [700, 65, 1536, 1, 300, 2000]
    probs = _problems(sizes, 2, KERNELS_2D, seed=7)
    out, info, alpha = _batch(probs)
    perm = [4, 2, 5, 0, 3, 1]
    outp, infop, _ = _batch([probs[i] for i in perm])
    for k, i in enumerate(perm):
        assert torch.equal(outp[k], out[i]) and int(infop[k]) == int(info[i])
    # other companions
    others = _problems([4096, 17, 900], 2, KERNELS_2D[::-1], seed=8)
    outc, _, _ = _batch([others[0], probs[2], others[1], probs[0], others[2]])
    assert torch.equal(outc[1], out[2]) and torch.equal(outc[3], out[0])
    # one problem not positive definite: info > 0 and -inf for it, nothing changes for the others
    X, y, e2, d = probs[4]
    e2bad = e2.clone()
    e2bad[37] = -1e3
    bad = list(probs)
    bad[4] = (X, y, e2bad, d)
    outb, infob, _ = _batch(bad)
    assert int(infob[4]) > 0 and float(outb[4, 0]) == -np.inf
    _, i1, _, _ = _single(bad[4])
    assert int(infob[4]) == int(i1.item())
    for b in range(len(probs)):
        if b != 4:
            assert torch.equal(outb[b], out[b]) and int(infob[b]) == 0


def test_chunking_and_repeatability(gpu_ready):
    from treegp_b200 import backend

    sizes = [400, 1200, 30, 2000, 513, 900, 64]
    probs = _problems(sizes, 2, KERNELS_2D, seed=9)
    out, info, alpha = _batch(probs)
    budget = 8 * backend.batch_work_doubles([2000]) + 1
    assert len(backend.plan_batch_chunks(sizes, budget)) >= 3
    outc, infoc, alphac = _batch(probs, budget=budget)
    assert torch.equal(outc, out) and torch.equal(infoc, info) and torch.equal(alphac, alpha)
    outa, _, alphaa = _batch(probs, want_alpha=True)
    for _ in range(20):
        o, i, a = _batch(probs)
        assert torch.equal(o, out) and torch.equal(i, info) and torch.equal(a, alpha)
    for _ in range(3):
        o, _, a = _batch(probs, want_alpha=True)
        assert torch.equal(o, outa) and torch.equal(a, alphaa)


def _api_data(B=6, seed=21):
    rng = np.random.default_rng(seed)
    sizes = np.linspace(300, 1500, B).astype(int)
    Xs, ys, es = [], [], []
    for n in sizes:
        X = rng.uniform(-15, 15, size=(n, 2))
        Xs.append(X)
        ys.append(np.sin(X[:, 0] / 3.0) * np.cos(X[:, 1] / 4.0) + rng.normal(scale=0.1, size=n) + 0.3)
        es.append(rng.uniform(0.05, 0.1, size=n))
    kstrs = ["%.2f * AnisotropicRBF(invLam=array([[%.3f, 0.0], [0.0, %.3f]]))" % (0.5 + 0.1 * b, 0.05 + 0.01 * b,
                                                                                    0.08 - 0.005 * b)
             for b in range(B)]
    Xn = [rng.uniform(-15, 15, size=(50 + 10 * b, 2)) for b in range(B)]
    return Xs, ys, es, kstrs, Xn


def _single_runs(optimizer, Xs, ys, es, kstrs, Xn, **kw):
    from treegp_b200 import GPInterpolation

    res = []
    for b in range(len(Xs)):
        gp = GPInterpolation(kernel=kstrs[b], optimizer=optimizer, **kw)
        gp.initialize(Xs[b], ys[b], y_err=es[b])
        gp.solve()
        res.append((gp.kernel.theta, gp.return_log_likelihood(), gp.predict(Xn[b])))
    return res


def test_api_log_likelihood_fit_matches_single_exactly(gpu_ready, monkeypatch):
    from treegp_b200 import GPInterpolation, GPInterpolationBatch, log_likelihood

    Xs, ys, es, kstrs, Xn = _api_data()
    gpb = GPInterpolationBatch(kernel=kstrs, optimizer="log-likelihood", white_noise=0.01)
    gpb.initialize(Xs, ys, es)
    gpb.solve()
    ll = gpb.return_log_likelihood()
    pred = gpb.predict(Xn)
    # defaults: the single path may take the envelope
    ref = _single_runs("log-likelihood", Xs, ys, es, kstrs, Xn, white_noise=0.01)
    for b in range(len(Xs)):
        np.testing.assert_allclose(gpb.kernels[b].theta, ref[b][0], rtol=1e-6)
        assert abs(ll[b] - ref[b][1]) <= 1e-9 * abs(ref[b][1])
    monkeypatch.setattr(log_likelihood, "BANDED", False)
    monkeypatch.setattr(GPInterpolation, "BANDED_SOLVE", False)
    ref = _single_runs("log-likelihood", Xs, ys, es, kstrs, Xn, white_noise=0.01)
    for b in range(len(Xs)):
        assert np.array_equal(gpb.kernels[b].theta, ref[b][0]), b
        assert ll[b] == ref[b][1], b
        np.testing.assert_allclose(pred[b], ref[b][2], rtol=1e-10, atol=1e-10 * np.max(np.abs(ref[b][2])))


@pytest.mark.parametrize("optimizer", ["none", "two-pcf", "anisotropic"])
def test_api_other_optimizers_match_single(gpu_ready, optimizer):
    from treegp_b200 import GPInterpolationBatch

    from treegp_b200 import GPInterpolation

    Xs, ys, es, kstrs, Xn = _api_data(B=3, seed=5)
    # Log binning (two-pcf) needs min_sep > 0; the anisotropic fit bins in TwoD from 0
    kw = {"none": {}, "two-pcf": dict(nbins=11, min_sep=0.5, max_sep=10.0),
          "anisotropic": dict(p0=[3.0, 0.0, 0.0], nbins=11, min_sep=0.0, max_sep=10.0)}[optimizer]
    gpb = GPInterpolationBatch(kernel=kstrs, optimizer=optimizer, **kw)
    gpb.initialize(Xs, ys, es)
    gpb.solve()
    ref = _single_runs(optimizer, Xs, ys, es, kstrs, Xn, **kw)
    pred = gpb.predict(Xn)
    for b in range(len(Xs)):
        if optimizer == "none":
            assert np.array_equal(gpb.kernels[b].theta, ref[b][0]), b
        else:
            # the batch runs the same per-problem 2PCF fit, but the pair sums are accumulated with FP64 atomics: two
            # single runs agree only to summation order, and so does the fitted theta (~1e-6 here)
            np.testing.assert_allclose(gpb.kernels[b].theta, ref[b][0], rtol=0, atol=1e-4)
        # predictions with the batch's fitted kernel against a single GP holding that kernel
        gp = GPInterpolation(kernel=kstrs[b], optimizer="none", **kw)
        gp.initialize(Xs[b], ys[b], y_err=es[b])
        gp.kernel = gpb.kernels[b]
        want = gp.predict(Xn[b])
        np.testing.assert_allclose(pred[b], want, rtol=1e-10, atol=1e-10 * np.max(np.abs(want)))


def test_api_not_positive_definite_names_the_problem(gpu_ready):
    """A problem whose matrix cannot be factorised (a NaN error: the pivot is not finite) gets -inf, the others are
    unaffected, and predict raises LinAlgError naming it."""
    from treegp_b200 import GPInterpolationBatch

    Xs, ys, es, kstrs, Xn = _api_data(B=3, seed=6)
    gpb = GPInterpolationBatch(kernel=kstrs, optimizer="none")
    gpb.initialize(Xs, ys, es)
    ll = gpb.return_log_likelihood()
    es[1] = es[1].copy()
    es[1][10] = np.nan
    gpb.initialize(Xs, ys, es)
    llb = gpb.return_log_likelihood()
    assert llb[1] == -np.inf and llb[0] == ll[0] and llb[2] == ll[2]
    with pytest.raises(np.linalg.LinAlgError, match="problem 1"):
        gpb.predict(Xn)
