"""GPU: the batched log-likelihood gradient (tgp_loglike_grad_batch) -- against tgp_loglike_grad_sum on each problem
alone (Z bit for bit, the values to 1e-12, the gradient to the rounding of alpha), against central differences of
the batched logL, independence of the problems, chunking and repeatability, failures, and GPInterpolationBatch's
analytic-gradient fit against per-problem GPInterpolation fits."""
import ctypes

import numpy as np
import pytest
import torch

from test_gpu_batch import KERNELS_1D, KERNELS_2D, SIZES, _problems

pytestmark = pytest.mark.gpu

# the finish's other column counts: one term with a white level (NC = 5), three and four terms (NC = 13, 17; the
# widest term grid of the sum contraction)
SUMS_2D = ["ConstantKernel(0.5) * RBF(4.0) + WhiteKernel(0.01)",
           "1.2 * AnisotropicRBF(invLam=array([[0.5, 0.1], [0.1, 0.8]])) + 0.4 * Matern(2.0, nu=1.5)"
           " + 0.3 * AnisotropicVonKarman(invLam=array([[0.9, -0.35], [-0.35, 0.6]])) + WhiteKernel(0.02)",
           "ConstantKernel(1.1) * RBF(0.9) + 0.4 * Matern(2.0, nu=0.5) + 0.3 * Matern(1.5, nu=2.5)"
           " + 0.2 * VonKarman(1.3) + WhiteKernel(0.03)"]
SUMS_1D = ["ConstantKernel(0.5) * RBF(4.0) + WhiteKernel(0.01)",
           "ConstantKernel(1.2) * RBF(0.9) + 0.4 * Matern(2.0, nu=1.5) + 0.3 * VonKarman(1.3)",
           "ConstantKernel(1.1) * RBF(0.9) + 0.4 * Matern(2.0, nu=0.5) + 0.3 * Matern(1.5, nu=2.5)"
           " + 0.2 * VonKarman(1.3) + WhiteKernel(0.03)"]


def _cat(probs):
    return (torch.cat([p[k] for p in probs]) for k in range(3))


def _grad_batch(probs, budget=4 << 30):
    from treegp_b200 import backend

    X, y, e2 = _cat(probs)
    return backend.loglike_grad_batch(X, y, e2, [p[0].shape[0] for p in probs], [p[3] for p in probs],
                                      budget_bytes=budget)


def _grad_batch_raw(probs):
    """One call of the C entry, keeping the workspace: (out, info, alpha, work)."""
    from treegp_b200 import _cabi, backend

    sizes = [p[0].shape[0] for p in probs]
    off = backend.batch_offsets(sizes)
    dev = probs[0][0].device
    work = torch.empty(backend.batch_work_doubles(sizes), dtype=torch.float64, device=dev)
    scratch = torch.empty(backend.grad_batch_scratch_doubles(sizes), dtype=torch.float64, device=dev)
    out = torch.empty((len(probs), _cabi.GRAD_BATCH_OUT), dtype=torch.float64, device=dev)
    info = torch.empty(len(probs), dtype=torch.int32, device=dev)
    alpha = torch.empty(int(off[-1]), dtype=torch.float64, device=dev)
    ks = backend._ksum_array([p[3] for p in probs])
    X, y, e2 = _cat(probs)
    _cabi.check(_cabi.load().tgp_loglike_grad_batch(
        backend._p(X), backend._p(y), backend._p(e2), backend._host_i64(off), len(probs),
        ctypes.cast(ks, ctypes.c_void_p), backend._p(work), backend._p(alpha), backend._p(out), backend._p(info),
        backend._p(scratch), backend._stream()), "tgp_loglike_grad_batch")
    return out, info, alpha, work


def _z_blocks(work, sizes):
    woff, blocks = 0, []
    for n in sizes:
        ld = (n + 1) // 2 * 2
        blocks.append(work[woff:woff + (n + 1) * ld].view(n + 1, ld)[:n, :n])
        woff += (n + 1) * ld
    return blocks


def _single(p):
    """tgp_loglike_grad_sum (dense) on one problem: (out, info, Z)."""
    from treegp_b200 import backend

    n = p[0].shape[0]
    out, info, _, work = backend.loglike_grad(p[0], p[1], p[2], backend.as_sum(p[3]))
    return out, info, work[:n, :n]


@pytest.mark.parametrize("ndim,kstrs,sums", [(2, KERNELS_2D, SUMS_2D), (1, KERNELS_1D, SUMS_1D)], ids=["2d", "1d"])
def test_grad_batch_against_single(gpu_ready, ndim, kstrs, sums):
    from treegp_b200 import backend

    # every size with every kernel: the sizes run through the kernel list at two offsets; then the other sums
    probs = (_problems(SIZES, ndim, kstrs, seed=30 + ndim) + _problems(SIZES, ndim, kstrs[3:] + kstrs[:3], seed=40)
             + _problems([2, 65, 513, 1536, 2000, 4096], ndim, sums, seed=50))
    sizes = [p[0].shape[0] for p in probs]
    ks = [backend.as_sum(p[3]) for p in probs]
    ncols = {4 if k.nterms == 1 and k.white == 0 else 4 * k.nterms + 1 for k in ks}   # the finish's NC
    assert ncols == {4, 5, 9, 13, 17}, ncols
    out, info, _, work = _grad_batch_raw(probs)
    Z = _z_blocks(work, sizes)
    for b, p in enumerate(probs):
        o1, i1, z1 = _single(p)
        k = o1.shape[0]
        assert int(info[b]) == 0 and int(i1.item()) == 0
        assert torch.equal(Z[b], z1), (b, sizes[b])
        for j in range(3):
            assert abs(float(out[b, j]) - float(o1[j])) <= 1e-12 * abs(float(o1[j])) + 1e-300, (b, j)
        g, g1 = out[b, 3:k], o1[3:]
        assert float((g - g1).abs().max()) <= 1e-9 * float(g1.abs().max()) + 1e-300, (b, sizes[b], g, g1)
        assert torch.all(out[b, k:] == 0)


def test_grad_batch_against_central_differences_of_the_batched_loglike(gpu_ready):
    from treegp_b200 import _cabi, backend

    sizes = [300, 700, 129]
    kstrs = ["1.5 * AnisotropicRBF(invLam=array([[0.5, 0.1], [0.1, 0.8]]))",
             "2.0 * AnisotropicVonKarman(invLam=array([[0.9, -0.35], [-0.35, 0.6]]))",
             "ConstantKernel(1.2) * RBF(0.9) + 0.4 * Matern(2.0, nu=1.5) + WhiteKernel(0.03)"]
    probs = _problems(sizes, 2, kstrs, seed=12)
    out, info, _ = _grad_batch(probs)
    X, y, e2 = _cat(probs)
    descs = [backend.as_sum(p[3]) for p in probs]
    h = 1e-5

    def logl(ds):
        o, _, _ = backend.loglike_batch(X, y, e2, sizes, ds)
        return o[:, 0].cpu().numpy()

    for b, d in enumerate(descs):
        k = 4 + 4 * d.nterms
        fd = []
        for c in range(d.nterms):
            for field in ("amp", "m00", "m01", "m11"):
                vals = []
                for sgn in (1.0, -1.0):
                    dd = _cabi.TgpKernelSum.from_buffer_copy(d)
                    t = dd.term[c]
                    if field == "amp":
                        t.amp = d.term[c].amp * np.exp(sgn * h)
                    else:
                        setattr(t, field, getattr(d.term[c], field) + sgn * h)
                    ds = list(descs)
                    ds[b] = dd
                    vals.append(logl(ds)[b])
                fd.append((vals[0] - vals[1]) / (2 * h))
        if d.white > 0:
            vals = []
            for sgn in (1.0, -1.0):
                dd = _cabi.TgpKernelSum.from_buffer_copy(d)
                dd.white = d.white * np.exp(sgn * h)
                ds = list(descs)
                ds[b] = dd
                vals.append(logl(ds)[b])
            fd.append((vals[0] - vals[1]) / (2 * h))
        g = out[b, 3:3 + len(fd)].cpu().numpy()
        np.testing.assert_allclose(g, fd, rtol=0, atol=1e-5 * np.max(np.abs(fd)) + 1e-6)
        assert int(info[b]) == 0 and np.all(out[b, k:].cpu().numpy() == 0)


def test_grad_batch_problems_are_independent_chunked_and_repeatable(gpu_ready):
    from treegp_b200 import backend

    sizes = [700, 65, 1536, 1, 300, 2000]
    probs = _problems(sizes, 2, KERNELS_2D, seed=7)
    out, info, alpha, work = _grad_batch_raw(probs)
    Z = _z_blocks(work, sizes)
    for b, p in enumerate(probs):   # alone
        o, i, _, w = _grad_batch_raw([p])
        assert torch.equal(o[0], out[b]) and int(i[0]) == int(info[b])
        assert torch.equal(_z_blocks(w, [sizes[b]])[0], Z[b])
    perm = [4, 2, 5, 0, 3, 1]
    outp, infop, _, workp = _grad_batch_raw([probs[i] for i in perm])
    Zp = _z_blocks(workp, [sizes[i] for i in perm])
    for k, i in enumerate(perm):
        assert torch.equal(outp[k], out[i]) and int(infop[k]) == int(info[i]) and torch.equal(Zp[k], Z[i])
    others = _problems([4096, 17, 900], 2, KERNELS_2D[::-1], seed=8)
    outc, _, _, workc = _grad_batch_raw([others[0], probs[2], others[1], probs[0], others[2]])
    Zc = _z_blocks(workc, [4096, 1536, 17, 700, 900])
    assert torch.equal(outc[1], out[2]) and torch.equal(outc[3], out[0])
    assert torch.equal(Zc[1], Z[2]) and torch.equal(Zc[3], Z[0])
    # chunks: the results do not depend on them
    outa, infoa, alphaa = _grad_batch(probs)
    budget = 8 * (backend.batch_work_doubles([2000]) + backend.grad_batch_scratch_doubles([2000])) + 1
    assert len(backend.plan_batch_chunks(sizes, budget, scratch=True)) >= 3
    outk, infok, alphak = _grad_batch(probs, budget=budget)
    assert torch.equal(outk, outa) and torch.equal(infok, infoa) and torch.equal(alphak, alphaa)
    assert torch.equal(outa, out) and torch.equal(alphaa, alpha)
    for _ in range(5):
        o, i, a, w = _grad_batch_raw(probs)
        assert torch.equal(o, out) and torch.equal(i, info) and torch.equal(a, alpha)
        assert all(torch.equal(z, zr) for z, zr in zip(_z_blocks(w, sizes), Z))


def test_grad_batch_not_positive_definite_and_non_finite(gpu_ready, monkeypatch):
    from treegp_b200 import GPInterpolationBatch, backend

    sizes = [700, 65, 1536, 300]
    probs = _problems(sizes, 2, KERNELS_2D, seed=17)
    out, info, _, work = _grad_batch_raw(probs)
    Z = _z_blocks(work, sizes)
    X, y, e2, d = probs[2]
    e2bad = e2.clone()
    e2bad[37] = -1e3
    bad = list(probs)
    bad[2] = (X, y, e2bad, d)
    outb, infob, _, workb = _grad_batch_raw(bad)
    Zb = _z_blocks(workb, sizes)
    o1, i1, _ = _single(bad[2])
    assert int(infob[2]) > 0 and int(infob[2]) == int(i1.item())
    assert float(outb[2, 0]) == -np.inf and torch.all(outb[2, 3:] == 0)
    for b in (0, 1, 3):
        assert torch.equal(outb[b], out[b]) and int(infob[b]) == 0 and torch.equal(Zb[b], Z[b])
    # non-finite descriptors: -inf and a zero gradient without a launch
    rng = np.random.default_rng(2)
    Xs = [rng.uniform(0, 20, size=(n, 2)) for n in (200, 300)]
    ys = [rng.normal(size=len(x)) for x in Xs]
    gpb = GPInterpolationBatch(kernel="1.5 * AnisotropicRBF(invLam=array([[0.5, 0.1], [0.1, 0.8]]))",
                               optimizer="log-likelihood")
    gpb.initialize(Xs, ys)
    calls = []
    real = backend.loglike_grad_batch
    monkeypatch.setattr(backend, "loglike_grad_batch", lambda *a, **k: calls.append(a[3]) or real(*a, **k))
    ks = [gpb.kernels[b].clone_with_theta(np.full_like(gpb.kernels[b].theta, np.nan)) for b in range(2)]
    res = gpb._loglike_and_gradient([0, 1], ks)
    assert not calls and all(v == -np.inf and np.all(g == 0) and len(g) == len(ks[0].theta) for v, g in res)
    res = gpb._loglike_and_gradient([0, 1], [ks[0], gpb.kernels[1]])
    assert calls == [[300]] and res[0][0] == -np.inf and np.isfinite(res[1][0]) and np.any(res[1][1] != 0)


def test_api_analytic_gradient_fit_matches_single(gpu_ready, monkeypatch):
    from treegp_b200 import GPInterpolation, GPInterpolationBatch, backend, log_likelihood

    rng = np.random.default_rng(31)
    sizes = [300, 520, 700, 900, 1100, 1300]
    Xs, ys, es = [], [], []
    for n in sizes:
        X = rng.uniform(-15, 15, size=(n, 2))
        Xs.append(X)
        ys.append(np.sin(X[:, 0] / 3.0) * np.cos(X[:, 1] / 4.0) + rng.normal(scale=0.1, size=n) + 0.3)
        es.append(rng.uniform(0.05, 0.1, size=n))
    kstrs = ["0.5 * AnisotropicRBF(invLam=array([[0.05, 0.0], [0.0, 0.08]]))",
             "0.6 * AnisotropicVonKarman(invLam=array([[0.04, 0.0], [0.0, 0.06]]))",
             "ConstantKernel(0.5) * RBF(4.0) + WhiteKernel(0.01)",
             "ConstantKernel(0.4) * Matern(5.0, nu=1.5)",
             "0.7 * AnisotropicRBF(invLam=array([[0.07, 0.0], [0.0, 0.05]]))",
             "ConstantKernel(0.5) * Matern(4.0, nu=2.5) + WhiteKernel(0.02)"]
    monkeypatch.setattr(log_likelihood, "BANDED", False)
    monkeypatch.setattr(GPInterpolation, "BANDED_SOLVE", False)
    counts = {"value": 0, "grad": 0}
    for name, key in (("loglike_batch", "value"), ("loglike_grad_batch", "grad")):
        real = getattr(backend, name)

        def wrapped(*a, _real=real, _key=key, **k):
            counts[_key] += 1
            return _real(*a, **k)
        monkeypatch.setattr(backend, name, wrapped)

    gpf = GPInterpolationBatch(kernel=kstrs, optimizer="log-likelihood")
    gpf.initialize(Xs, ys, es)
    gpf.solve()
    rounds_fd = counts["value"]
    monkeypatch.setattr(log_likelihood, "ANALYTIC_GRADIENT", True)
    counts.update(value=0, grad=0)
    gpb = GPInterpolationBatch(kernel=kstrs, optimizer="log-likelihood")
    gpb.initialize(Xs, ys, es)
    gpb.solve()
    rounds_an = counts["grad"]
    assert counts["value"] == 0 and 0 < rounds_an < rounds_fd, (rounds_an, rounds_fd)
    ll = gpb.return_log_likelihood()
    for b in range(len(Xs)):
        gp = GPInterpolation(kernel=kstrs[b], optimizer="log-likelihood")
        gp.initialize(Xs[b], ys[b], y_err=es[b])
        gp.solve()
        np.testing.assert_allclose(gpb.kernels[b].theta, gp.kernel.theta, rtol=1e-6)
        ref = gp.return_log_likelihood()
        assert abs(ll[b] - ref) <= 1e-9 * abs(ref), b
