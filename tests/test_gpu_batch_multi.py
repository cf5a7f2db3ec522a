"""GPU: several outputs per problem in a batch (tgp_loglike_batch_multi, tgp_loglike_grad_batch_multi,
tgp_predict_mean_batch_multi, tgp_loo_batch_multi) -- bit for bit against tgp_loglike_multi on each problem alone and
against the single-output batch column by column, the joint gradient against tgp_loglike_grad_multi and the numpy
oracle, independence of the problems, of chunking and of repeats, and GPInterpolationBatch with 2-D ys against
per-problem multi-output GPInterpolation."""
import ctypes

import numpy as np
import pytest
import torch

import multi_oracle as mo
import sum_oracle as so
from test_gpu_batch import KERNELS_1D, KERNELS_2D, SIZES, _problems

pytestmark = pytest.mark.gpu

RS = [1, 2, 3, 8]


def _with_outputs(probs, r, seed):
    """The problems with Y (N, r) in place of y (N,)."""
    from treegp_b200 import backend

    rng = np.random.default_rng(seed)
    return [(X, backend.to_device(rng.normal(size=(X.shape[0], r))), e2, d) for X, _, e2, d in probs]


def _cat(probs):
    return tuple(torch.cat([p[k] for p in probs]) for k in range(3))


def _sizes(probs):
    return [p[0].shape[0] for p in probs]


def _raw_loglike(probs, r, want_alpha):
    """One tgp_loglike_batch_multi call with a workspace of its own: (out, info, alpha, work, offsets)."""
    from treegp_b200 import _cabi, backend

    sizes = _sizes(probs)
    off = backend.batch_offsets(sizes)
    dev = probs[0][0].device
    X, Y, e2 = _cat(probs)
    work = torch.empty(int(_cabi.load().tgp_batch_multi_work_doubles(backend._host_i64(off), len(probs), r)),
                       dtype=torch.float64, device=dev)
    assert work.numel() == backend.batch_work_doubles(sizes, r)
    out = torch.empty((len(probs), 3), dtype=torch.float64, device=dev)
    info = torch.empty(len(probs), dtype=torch.int32, device=dev)
    alpha = torch.empty(Y.shape, dtype=torch.float64, device=dev)
    ks = backend._ksum_array([p[3] for p in probs])
    _cabi.check(_cabi.load().tgp_loglike_batch_multi(
        backend._p(X), backend._p(Y), r, backend._p(e2), backend._host_i64(off), len(probs),
        ctypes.cast(ks, ctypes.c_void_p), backend._p(work), backend._p(alpha), int(want_alpha), backend._p(out),
        backend._p(info), backend._stream()), "tgp_loglike_batch_multi")
    return out, info, alpha, work, off


@pytest.mark.parametrize("r", RS)
@pytest.mark.parametrize("ndim,kstrs", [(2, KERNELS_2D), (1, KERNELS_1D)], ids=["2d", "1d"])
def test_loglike_batch_multi_bitwise_against_single(gpu_ready, ndim, kstrs, r):
    from treegp_b200 import backend

    probs = _with_outputs(_problems(SIZES, ndim, kstrs, seed=110 + ndim), r, seed=120 + r)
    sizes = _sizes(probs)
    out, info, alpha, work, off = _raw_loglike(probs, r, want_alpha=False)
    woff = 0
    for b, p in enumerate(probs):
        n, ld = sizes[b], (sizes[b] + 1) // 2 * 2
        o1, i1, a1, w1 = backend.loglike(p[0], p[1], p[2], p[3])   # tgp_loglike_multi, dense
        assert int(info[b]) == 0 and int(i1.item()) == 0
        assert torch.equal(out[b], o1), (b, n, out[b], o1)
        assert torch.equal(alpha[off[b]:off[b + 1]], a1), (b, n)
        blk = work[woff:woff + (n + r) * ld].view(n + r, ld)
        assert torch.equal(torch.tril(blk[:n, :n]), torch.tril(w1[:n, :n])), (b, n)
        assert torch.equal(blk[n:n + r, :n], w1[n:n + r, :n]), (b, n)   # L^-1 Y
        woff += (n + r) * ld
    # the backend function gives the same, and alpha = K^-1 Y column by column as the single-output batch
    X, Y, e2 = _cat(probs)
    descs = [p[3] for p in probs]
    outb, infob, alphab = backend.loglike_batch(X, Y, e2, sizes, descs)
    assert torch.equal(outb, out) and torch.equal(infob, info) and torch.equal(alphab, alpha)
    outa, infoa, alphaa = backend.loglike_batch(X, Y, e2, sizes, descs, want_alpha=True)
    assert torch.equal(infoa, info)
    assert torch.equal(outa[:, 2], out[:, 2])
    for c in range(r):
        _, _, ac = backend.loglike_batch(X, Y[:, c].contiguous(), e2, sizes, descs, want_alpha=True)
        assert torch.equal(alphaa[:, c], ac), c
    if r == 1:   # (sum N, 1) is the 1-D path bit for bit
        for wa in (False, True):
            o1, i1, a1 = backend.loglike_batch(X, Y[:, 0].contiguous(), e2, sizes, descs, want_alpha=wa)
            o2, i2, a2 = backend.loglike_batch(X, Y, e2, sizes, descs, want_alpha=wa)
            assert torch.equal(o1, o2) and torch.equal(i1, i2) and torch.equal(a1, a2[:, 0]) and a2.shape == Y.shape


@pytest.mark.parametrize("r", [2, 3, 8])
@pytest.mark.parametrize("ndim,kstrs", [(2, KERNELS_2D), (1, KERNELS_1D)], ids=["2d", "1d"])
def test_loglike_grad_batch_multi_against_single_and_oracle(gpu_ready, ndim, kstrs, r):
    from treegp_b200 import _cabi, backend

    sizes = [1, 63, 65, 513, 1536, 2000] if r != 8 else SIZES
    probs = _with_outputs(_problems(sizes, ndim, kstrs, seed=130 + ndim), r, seed=140 + r)
    X, Y, e2 = _cat(probs)
    descs = [p[3] for p in probs]
    out, info, alpha = backend.loglike_grad_batch(X, Y, e2, sizes, descs)
    outv, _, alphav = backend.loglike_batch(X, Y, e2, sizes, descs, want_alpha=True)
    assert torch.equal(out[:, :3], outv) and torch.equal(alpha, alphav)
    off = backend.batch_offsets(sizes)
    for b, p in enumerate(probs):
        assert int(info[b]) == 0
        ks = backend.as_sum(p[3])
        n_out = 4 + 4 * ks.nterms
        o1, i1, _, _ = backend.loglike_grad(p[0], p[1], p[2], p[3])   # tgp_loglike_grad_multi, dense
        g, g1 = out[b, 3:n_out], o1[3:n_out]
        scale = float(g1.abs().max())
        assert float((g - g1).abs().max()) <= 1e-9 * scale, (b, sizes[b], g, g1)
        assert abs(float(out[b, 0]) - float(o1[0])) <= 1e-12 * abs(float(o1[0]))
        assert torch.equal(out[b, n_out:], torch.zeros_like(out[b, n_out:]))
        if sizes[b] <= 200:
            terms, white = so.terms_of(ks)
            ll, go, A = mo.joint_log_likelihood_gradient(terms, white, p[0].cpu().numpy(), p[1].cpu().numpy(),
                                                         p[2].cpu().numpy())
            assert abs(float(out[b, 0]) - ll) <= 1e-9 * abs(ll)
            assert np.max(np.abs(g.cpu().numpy() - go)) <= 1e-9 * np.max(np.abs(go)), (b, sizes[b])
            np.testing.assert_allclose(alpha[off[b]:off[b + 1]].cpu().numpy(), A, rtol=1e-8,
                                       atol=1e-10 * np.max(np.abs(A)))
    # Z = K^-1 in the workspace equals tgp_selinv on the dense factor of tgp_loglike_multi bit for bit
    lib = _cabi.load()
    work = torch.empty(backend.batch_work_doubles(sizes, r), dtype=torch.float64, device=gpu_ready)
    scratch = torch.empty(backend.grad_batch_scratch_doubles(sizes), dtype=torch.float64, device=gpu_ready)
    o2 = torch.empty((len(sizes), _cabi.GRAD_BATCH_OUT), dtype=torch.float64, device=gpu_ready)
    i2 = torch.empty(len(sizes), dtype=torch.int32, device=gpu_ready)
    a2 = torch.empty(Y.shape, dtype=torch.float64, device=gpu_ready)
    ksa = backend._ksum_array(descs)
    _cabi.check(lib.tgp_loglike_grad_batch_multi(
        backend._p(X), backend._p(Y), r, backend._p(e2), backend._host_i64(off), len(sizes),
        ctypes.cast(ksa, ctypes.c_void_p), backend._p(work), backend._p(a2), backend._p(o2), backend._p(i2),
        backend._p(scratch), backend._stream()), "tgp_loglike_grad_batch_multi")
    assert torch.equal(o2, out)
    woff = 0
    for b, p in enumerate(probs):
        n, ld = sizes[b], (sizes[b] + 1) // 2 * 2
        _, _, _, w1 = backend.loglike(p[0], p[1], p[2], p[3])
        backend.selinv(w1, n)
        blk = work[woff:woff + (n + r) * ld].view(n + r, ld)
        assert torch.equal(blk[:n, :n], w1[:n, :n]), (b, n)
        woff += (n + r) * ld


@pytest.mark.parametrize("r", RS)
def test_predict_mean_batch_multi_equals_single(gpu_ready, r):
    from treegp_b200 import backend

    sizes = [1, 63, 200, 256, 700, 2000]
    probs = _with_outputs(_problems(sizes, 2, KERNELS_2D, seed=150), r, seed=151 + r)
    X, Y, e2 = _cat(probs)
    descs = [p[3] for p in probs]
    _, _, alpha = backend.loglike_batch(X, Y, e2, sizes, descs, want_alpha=True)
    off = backend.batch_offsets(sizes)
    rng = np.random.default_rng(152)
    ssizes = [5, 0, 257, 40, 1, 600]
    Xs = [backend.to_device(rng.uniform(0, 60, size=(m, 2))) for m in ssizes]
    mean = backend.predict_mean_batch(torch.cat(Xs), ssizes, X, sizes, descs, alpha)
    assert mean.shape == (sum(ssizes), r)
    soff = backend.batch_offsets(ssizes)
    R = 1 if r == 1 else 2 if r <= 2 else 4 if r <= 4 else 8
    tile = 1024 if R == 1 else 2048 // R
    for b, p in enumerate(probs):
        if ssizes[b] == 0:
            continue
        ref = backend.predict_mean(Xs[b], p[0], p[3], alpha[off[b]:off[b + 1]].contiguous(), truncate=False)
        got = mean[soff[b]:soff[b + 1]]
        if sizes[b] <= tile:   # the single call runs unsplit: the same sum bit for bit
            assert torch.equal(got, ref), (b, r)
        else:                  # the single call splits the training tiles over CTAs (atomic partial sums)
            assert float((got - ref).abs().max()) <= 1e-12 * float(ref.abs().max())
    if r == 1:
        m1 = backend.predict_mean_batch(torch.cat(Xs), ssizes, X, sizes, descs, alpha[:, 0].contiguous())
        assert torch.equal(m1, mean[:, 0])


@pytest.mark.parametrize("r", [1, 2, 8])
def test_loo_batch_multi_columns_and_failures(gpu_ready, r):
    from treegp_b200 import backend

    sizes = [1, 64, 513, 2000, 300]
    probs = _with_outputs(_problems(sizes, 2, KERNELS_2D, seed=160), r, seed=161 + r)
    X, Y, e2 = _cat(probs)
    descs = [p[3] for p in probs]
    mean, var, info = backend.loo_batch(X, Y, e2, sizes, descs)
    assert torch.all(info == 0) and mean.shape == Y.shape and var.shape == (X.shape[0],)
    for c in range(r):   # each output as the single-output batch: the same alpha column and Z
        mc, vc, _ = backend.loo_batch(X, Y[:, c].contiguous(), e2, sizes, descs)
        assert torch.equal(mean[:, c], mc), c
        assert torch.equal(var, vc)
    # a problem that is not positive definite: NaN rows for it alone
    e2bad = e2.clone()
    off = backend.batch_offsets(sizes)
    e2bad[int(off[4]) + 37] = -1e3
    meanb, varb, infob = backend.loo_batch(X, Y, e2bad, sizes, descs)
    assert int(infob[4]) > 0
    assert torch.all(torch.isnan(meanb[off[4]:])) and torch.all(torch.isnan(varb[off[4]:]))
    assert torch.equal(meanb[:off[4]], mean[:off[4]]) and torch.equal(varb[:off[4]], var[:off[4]])


def test_batch_multi_independent_of_order_subsets_chunking_and_repeats(gpu_ready):
    from treegp_b200 import backend

    r = 3
    sizes = [700, 65, 1536, 1, 2000, 300]
    probs = _with_outputs(_problems(sizes, 2, KERNELS_2D, seed=170), r, seed=171)

    def run(ps, **kw):
        X, Y, e2 = _cat(ps)
        return backend.loglike_batch(X, Y, e2, _sizes(ps), [p[3] for p in ps], **kw)

    out, info, alpha = run(probs, want_alpha=True)
    off = backend.batch_offsets(sizes)
    perm = [4, 2, 5, 0, 3, 1]
    outp, infop, alphap = run([probs[i] for i in perm], want_alpha=True)
    offp = backend.batch_offsets([sizes[i] for i in perm])
    for k, i in enumerate(perm):
        assert torch.equal(outp[k], out[i]) and int(infop[k]) == int(info[i])
        assert torch.equal(alphap[offp[k]:offp[k + 1]], alpha[off[i]:off[i + 1]])
    outs, _, _ = run([probs[2], probs[0]], want_alpha=True)
    assert torch.equal(outs[0], out[2]) and torch.equal(outs[1], out[0])
    budget = 8 * backend.batch_work_doubles([2000], r) + 1
    assert len(backend.plan_batch_chunks(sizes, budget, r=r)) >= 3
    outc, infoc, alphac = run(probs, want_alpha=True, budget_bytes=budget)
    assert torch.equal(outc, out) and torch.equal(infoc, info) and torch.equal(alphac, alpha)
    X, Y, e2 = _cat(probs)
    descs = [p[3] for p in probs]
    g, _, _ = backend.loglike_grad_batch(X, Y, e2, sizes, descs)
    gc, _, _ = backend.loglike_grad_batch(X, Y, e2, sizes, descs, budget_bytes=budget)
    assert torch.equal(g, gc)
    for _ in range(3):
        o, i, a = run(probs, want_alpha=True)
        assert torch.equal(o, out) and torch.equal(a, alpha)
        assert torch.equal(backend.loglike_grad_batch(X, Y, e2, sizes, descs)[0], g)


def _api_data(B=4, r=2, seed=31):
    rng = np.random.default_rng(seed)
    sizes = np.linspace(300, 1200, B).astype(int)
    Xs, ys, es = [], [], []
    for n in sizes:
        X = rng.uniform(-15, 15, size=(n, 2))
        Xs.append(X)
        base = np.sin(X[:, 0] / 3.0) * np.cos(X[:, 1] / 4.0)
        ys.append(np.stack([base * (1.0 + 0.3 * c) + rng.normal(scale=0.1, size=n) + 0.2 * c for c in range(r)],
                           axis=1))
        es.append(rng.uniform(0.05, 0.1, size=n))
    kstrs = ["%.2f * AnisotropicRBF(invLam=array([[%.3f, 0.0], [0.0, %.3f]]))" % (0.5 + 0.1 * b, 0.05 + 0.01 * b,
                                                                                    0.08 - 0.005 * b)
             for b in range(B)]
    Xn = [rng.uniform(-15, 15, size=(40 + 10 * b, 2)) for b in range(B)]
    return Xs, ys, es, kstrs, Xn


def test_api_multi_output_matches_single(gpu_ready, monkeypatch):
    from treegp_b200 import GPInterpolation, GPInterpolationBatch, log_likelihood

    monkeypatch.setattr(log_likelihood, "BANDED", False)
    monkeypatch.setattr(GPInterpolation, "BANDED_SOLVE", False)
    Xs, ys, es, kstrs, Xn = _api_data()
    gpb = GPInterpolationBatch(kernel=kstrs, optimizer="log-likelihood", white_noise=0.01)
    gpb.initialize(Xs, ys, es)
    gpb.solve()
    ll = gpb.return_log_likelihood()
    pred = gpb.predict(Xn)
    pm, pv = gpb.predict_var(Xn)
    lm, lv = gpb.loo_predict()
    for b in range(len(Xs)):
        gp = GPInterpolation(kernel=kstrs[b], optimizer="log-likelihood", white_noise=0.01)
        gp.initialize(Xs[b], ys[b], y_err=es[b])
        gp.solve()
        assert np.array_equal(gpb.kernels[b].theta, gp.kernel.theta), b
        assert ll[b] == gp.return_log_likelihood(), b
        ref = gp.predict(Xn[b])
        assert pred[b].shape == ref.shape == (len(Xn[b]), 2)
        np.testing.assert_allclose(pred[b], ref, rtol=1e-10, atol=1e-10 * np.max(np.abs(ref)))
        rm, rv = gp.predict_var(Xn[b])
        assert pm[b].shape == rm.shape and pv[b].shape == rv.shape == (len(Xn[b]),)
        np.testing.assert_array_equal(pm[b], pred[b])
        gp.WINDOWED_VARIANCE = False
        _, rv = gp.predict_var(Xn[b])
        assert np.array_equal(pv[b], rv), b
        rlm, rlv = gp.loo_predict()
        assert lm[b].shape == rlm.shape == ys[b].shape
        np.testing.assert_allclose(lm[b], rlm, rtol=1e-9, atol=1e-9 * np.max(np.abs(rlm)))
        assert np.array_equal(lv[b], rlv), b
    # the analytic gradient: the per-problem optimum to 1e-6
    monkeypatch.setattr(log_likelihood, "ANALYTIC_GRADIENT", True)
    gpa = GPInterpolationBatch(kernel=kstrs, optimizer="log-likelihood", white_noise=0.01)
    gpa.initialize(Xs, ys, es)
    gpa.solve()
    for b in range(len(Xs)):
        gp = GPInterpolation(kernel=kstrs[b], optimizer="log-likelihood", white_noise=0.01)
        gp.initialize(Xs[b], ys[b], y_err=es[b])
        gp.solve()
        np.testing.assert_allclose(gpa.kernels[b].theta, gp.kernel.theta, rtol=1e-6, atol=1e-6)


def test_api_multi_output_shapes_and_errors(gpu_ready):
    from treegp_b200 import GPInterpolationBatch

    Xs, ys, es, kstrs, Xn = _api_data(B=3, r=1, seed=33)
    gp = GPInterpolationBatch(kernel=kstrs, optimizer="none")
    gp.initialize(Xs, ys, es)   # (N_b, 1): (., 1) shapes back
    assert all(p.shape == (len(x), 1) for p, x in zip(gp.predict(Xn), Xn))
    m, v = gp.loo_predict()
    assert all(a.shape == (len(x), 1) and w.shape == (len(x),) for a, w, x in zip(m, v, Xs))
    g1 = GPInterpolationBatch(kernel=kstrs, optimizer="none")
    g1.initialize(Xs, [y[:, 0] for y in ys], es)
    for a, b in zip(gp.predict(Xn), g1.predict(Xn)):
        assert np.array_equal(a[:, 0], b)
    assert np.array_equal(gp.return_log_likelihood(), g1.return_log_likelihood())
    with pytest.raises(ValueError, match="two-pcf / anisotropic"):
        bad = GPInterpolationBatch(kernel=kstrs, optimizer="two-pcf")
        bad.initialize(Xs, ys, es)
        bad.solve()
    # the failing problem is named
    gp2 = GPInterpolationBatch(kernel=kstrs, optimizer="none")
    gp2.initialize(Xs, ys, es)
    gp2.kernels[1] = gp2.kernels[1].clone_with_theta(np.full(len(gp2.kernels[1].theta), np.nan))
    for call in (gp2.loo_predict, lambda: gp2.predict(Xn), lambda: gp2.predict_var(Xn)):
        with pytest.raises(np.linalg.LinAlgError, match="problem 1"):
            call()
    # a problem that is not positive definite with 2-D ys: named from the device's info, nothing raised for the others
    Xs2, ys2, es2, kstrs2, Xn2 = _api_data(B=3, r=2, seed=34)
    gp3 = GPInterpolationBatch(kernel=kstrs2, optimizer="none")
    gp3.initialize(Xs2, ys2, es2)
    _, _, e2, _, off = gp3._device_data()
    e2[int(off[1]) + 37] = -1e3
    for call in (gp3.loo_predict, lambda: gp3.predict(Xn2), lambda: gp3.predict_var(Xn2)):
        with pytest.raises(np.linalg.LinAlgError, match="problem 1: .* not positive definite"):
            call()
    ll = gp3.return_log_likelihood()
    assert ll[1] == -np.inf and np.all(np.isfinite(ll[[0, 2]]))
    with pytest.raises(ValueError, match="means only"):
        gp.predict(Xn, return_cov=True)
