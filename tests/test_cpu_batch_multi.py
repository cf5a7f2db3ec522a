"""CPU: several outputs per problem in a batch without a GPU -- argument validation of the _multi batch entries
(tgp_batch_multi_work_doubles, tgp_loglike_batch_multi, tgp_loglike_grad_batch_multi, tgp_predict_mean_batch_multi,
tgp_loo_batch_multi), the workspace formula, the chunk planner with r outputs, and GPInterpolationBatch rejecting
malformed 2-D input before any device work."""
import ctypes

import numpy as np
import pytest

P16 = ctypes.c_void_p(16)


def _lib():
    from treegp_b200 import _cabi

    return _cabi, _cabi.load()


def _sums(B, family=0, ndim=2):
    _cabi, _ = _lib()
    arr = (_cabi.TgpKernelSum * B)()
    for b in range(B):
        arr[b].nterms, arr[b].ndim, arr[b].white = 1, ndim, 0.0
        arr[b].term[0] = _cabi.TgpKernel(family, ndim, 1.0, 1.0, 0.0, 1.0)
    return arr


def _off(sizes):
    return np.ascontiguousarray(np.concatenate([[0], np.cumsum(sizes)]), dtype=np.int64)


def _ptr(a):
    return None if a is None else ctypes.c_void_p(a.ctypes.data)


def _calls(lib, off, B, ks, r, X=P16, Y=P16, e2=P16, work=P16, alpha=P16, out=P16, info=P16, scratch=P16, Xs=P16,
           soff=None, mean=P16, var=P16):
    soff = _off([3] * B) if soff is None else soff
    return {
        "tgp_loglike_batch_multi": lambda: lib.tgp_loglike_batch_multi(X, Y, r, e2, _ptr(off), B, ks, work, alpha, 0,
                                                                       out, info, None),
        "tgp_loglike_grad_batch_multi": lambda: lib.tgp_loglike_grad_batch_multi(X, Y, r, e2, _ptr(off), B, ks, work,
                                                                                 alpha, out, info, scratch, None),
        "tgp_predict_mean_batch_multi": lambda: lib.tgp_predict_mean_batch_multi(Xs, _ptr(soff), X, _ptr(off), B, ks,
                                                                                 alpha, r, mean, None),
        "tgp_loo_batch_multi": lambda: lib.tgp_loo_batch_multi(X, Y, r, e2, _ptr(off), B, ks, work, alpha, scratch,
                                                               mean, var, info, None),
    }


def test_multi_batch_entries_reject_bad_arguments_without_a_gpu():
    _, lib = _lib()
    off, ks = _off([10, 20, 30]), _sums(3)
    for r, msg in ((0, b"number of outputs r must be 1 .. TGP_MAX_RHS"), (9, b"number of outputs r")):
        for name, call in _calls(lib, off, 3, ks, r).items():
            assert call() == -1, (name, r)
            err = lib.tgp_last_error()
            assert err.startswith(name.encode() + b": invalid argument") and msg in err, (name, err)
        assert lib.tgp_batch_multi_work_doubles(_ptr(off), 3, r) == -1
        assert b"number of outputs" in lib.tgp_last_error()
    cases = [(dict(B=0), b"B must be >= 1"), (dict(off=None), b"off must be a host array"),
             (dict(off=_off([10, 0, 30])), b"strictly increasing"), (dict(off=_off([10, 4097, 30])), b"TGP_BATCH_MAX_N"),
             (dict(ks=None), b"ks")]
    for kw, msg in cases:
        a = dict(off=off, B=3, ks=ks)
        a.update(kw)
        for name, call in _calls(lib, a["off"], a["B"], a["ks"], 2).items():
            assert call() == -1, (name, msg)
            err = lib.tgp_last_error()
            assert err.startswith(name.encode() + b": invalid argument") and msg in err, (name, err)
    # null pointers (Y among them) and misaligned work or scratch, for every entry that takes them
    for name in ("X", "Y", "e2", "work", "alpha", "out", "info", "scratch", "mean", "var", "Xs"):
        for entry, call in _calls(lib, off, 3, ks, 2, **{name: None}).items():
            needs = {"tgp_loglike_batch_multi": "X Y e2 work alpha out info",
                     "tgp_loglike_grad_batch_multi": "X Y e2 work alpha out info scratch",
                     "tgp_predict_mean_batch_multi": "Xs X alpha mean",
                     "tgp_loo_batch_multi": "X Y e2 work alpha scratch mean var info"}[entry].split()
            if name in needs:
                assert call() == -1, (entry, name)
                assert b"null pointer" in lib.tgp_last_error(), (entry, name)
    for name in ("work", "scratch"):
        for entry, call in _calls(lib, off, 3, ks, 2, **{name: ctypes.c_void_p(24)}).items():
            if entry == "tgp_predict_mean_batch_multi" or (name == "scratch" and entry == "tgp_loglike_batch_multi"):
                continue
            assert call() == -1, (entry, name)
            assert (name + " must be 16-byte aligned").encode() in lib.tgp_last_error(), (entry, name)
    # no test points: nothing to do
    assert lib.tgp_predict_mean_batch_multi(P16, _ptr(_off([0, 0, 0])), P16, _ptr(off), 3, ks, P16, 8, P16, None) == 0


def test_multi_workspace_formula_and_chunk_plan():
    from treegp_b200 import backend

    _, lib = _lib()
    sizes = [1, 2, 63, 511, 4096]
    off = _off(sizes)
    for r in range(1, 9):
        want = sum((n + r) * ((n + 1) // 2 * 2) for n in sizes)
        assert lib.tgp_batch_multi_work_doubles(_ptr(off), len(sizes), r) == want == backend.batch_work_doubles(sizes, r)
    assert lib.tgp_batch_multi_work_doubles(_ptr(off), len(sizes), 1) == lib.tgp_batch_work_doubles(_ptr(off), len(sizes))
    assert backend.batch_work_doubles(sizes) == backend.batch_work_doubles(sizes, 1)
    rng = np.random.default_rng(5)
    for _ in range(200):
        B = int(rng.integers(1, 20))
        sz = [int(n) for n in rng.integers(1, 4097, size=B)]
        r = int(rng.integers(1, 9))
        scratch = bool(rng.integers(0, 2))
        budget = int(rng.integers(1 << 18, 1 << 30))
        chunks = backend.plan_batch_chunks(sz, budget, scratch=scratch, r=r)
        assert chunks[0][0] == 0 and chunks[-1][1] == B
        assert all(a[1] == b[0] for a, b in zip(chunks, chunks[1:]))
        for b0, b1 in chunks:
            need = 8 * backend.batch_work_doubles(sz[b0:b1], r)
            if scratch:
                need += 8 * backend.grad_batch_scratch_doubles(sz[b0:b1])
            assert b1 - b0 == 1 or need <= budget
    assert backend.plan_batch_chunks([4096] * 4, 8 * backend.batch_work_doubles([4096] * 2)) == [(0, 2), (2, 4)]
    assert len(backend.plan_batch_chunks([4096] * 4, 8 * backend.batch_work_doubles([4096] * 2), r=8)) == 4


def test_gp_batch_rejects_bad_multi_output_input_before_device_work(monkeypatch):
    from treegp_b200 import GPInterpolationBatch, backend

    def no_device(*a, **k):
        raise AssertionError("device touched")

    for name in ("loglike_batch", "loglike_grad_batch", "predict_mean_batch", "predict_var_batch", "loo_batch",
                 "as_points", "to_device"):
        monkeypatch.setattr(backend, name, no_device)
    rng = np.random.default_rng(0)
    Xs = [rng.uniform(size=(n, 2)) for n in (30, 40)]
    gp = GPInterpolationBatch(kernel="RBF(1.0)", optimizer="none")
    with pytest.raises(ValueError, match="1-D"):
        gp.initialize(Xs, [rng.normal(size=(30, 2)), rng.normal(size=40)])
    with pytest.raises(ValueError, match="one r"):
        gp.initialize(Xs, [rng.normal(size=(30, 2)), rng.normal(size=(40, 3))])
    with pytest.raises(ValueError, match="TGP_MAX_RHS"):
        gp.initialize(Xs, [rng.normal(size=(30, 9)), rng.normal(size=(40, 9))])
    with pytest.raises(ValueError, match="TGP_MAX_RHS"):
        gp.initialize(Xs, [rng.normal(size=(30, 0)), rng.normal(size=(40, 0))])
    with pytest.raises(ValueError, match=r"y_err must have shape \(N,\)"):
        gp.initialize(Xs, [rng.normal(size=(30, 2)), rng.normal(size=(40, 2))], [np.ones((30, 2)), np.ones(40)])
    with pytest.raises(ValueError, match="1-D"):
        gp.initialize(Xs, [rng.normal(size=(30, 2, 1)), rng.normal(size=(40, 2, 1))])
    ys = [rng.normal(size=(30, 3)), rng.normal(size=(40, 3))]
    gp.initialize(Xs, ys, [np.full(30, 0.1), None])
    # one normalising mean per output, column by column
    assert gp._mean[0].shape == (3,)
    assert all(gp._mean[0][c] == np.mean(np.ascontiguousarray(ys[0][:, c])) for c in range(3))
    with pytest.raises(ValueError, match="means only"):
        gp.predict(Xs, return_cov=True)
    for opt in ("two-pcf", "anisotropic"):
        g2 = GPInterpolationBatch(kernel="RBF(1.0)", optimizer=opt)
        g2.initialize(Xs, ys)
        with pytest.raises(ValueError, match="need a 1-D y; with several outputs"):
            g2.solve()
