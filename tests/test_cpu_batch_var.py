"""CPU: predictive variance and leave-one-out predictions of a batch without a GPU -- argument validation of
tgp_predict_var_batch, its workspace size and tgp_loo_batch, GPInterpolationBatch.predict_var / loo_predict rejecting
malformed input before any device work, and the host planner of test points per pass."""
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


def _var(lib, soff, off, B, ks, chunk=64, Xs=P16, X=P16, work=P16, vwork=P16, var=P16):
    return lib.tgp_predict_var_batch(Xs, _ptr(soff), X, _ptr(off), B, ks, work, vwork, chunk, var, None)


def _loo(lib, off, B, ks, X=P16, y=P16, e2=P16, work=P16, alpha=P16, scratch=P16, mean=P16, var=P16, info=P16):
    return lib.tgp_loo_batch(X, y, e2, _ptr(off), B, ks, work, alpha, scratch, mean, var, info, None)


def test_var_batch_entries_reject_bad_arguments_without_a_gpu():
    _, lib = _lib()
    off, soff = _off([10, 20, 30]), _off([5, 0, 7])
    ks = _sums(3)
    cases = [
        (dict(B=0), b"B must be >= 1"),
        (dict(off=None), b"off must be a host array"),
        (dict(soff=None), b"soff must be a host array"),
        (dict(off=_off([10, 0, 30])), b"off must be strictly increasing"),
        (dict(off=_off([10, 4097, 30])), b"TGP_BATCH_MAX_N"),
        (dict(soff=np.array([0, 5, 3, 9], dtype=np.int64)), b"soff must be non-decreasing"),
        (dict(soff=np.array([2, 5, 6, 9], dtype=np.int64)), b"soff[0] must be 0"),
        (dict(chunk=0), b"chunk must be >= 1"),
        (dict(ks=None), b"ks"),
    ]
    for kw, msg in cases:
        a = dict(soff=soff, off=off, B=3, ks=ks)
        a.update(kw)
        assert _var(lib, a["soff"], a["off"], a["B"], a["ks"], chunk=a.get("chunk", 64)) == -1, msg
        err = lib.tgp_last_error()
        assert err.startswith(b"tgp_predict_var_batch: invalid argument") and msg in err, (msg, err)
    for name in ("X", "work", "Xs", "vwork", "var"):
        assert _var(lib, soff, off, 3, ks, **{name: None}) == -1, name
        assert b"null pointer" in lib.tgp_last_error()
    assert _var(lib, soff, off, 3, ks, work=ctypes.c_void_p(24)) == -1
    assert b"work must be 16-byte" in lib.tgp_last_error()
    assert _var(lib, soff, off, 3, ks, vwork=ctypes.c_void_p(24)) == -1
    assert b"vwork must be 16-byte" in lib.tgp_last_error()
    # no test points at all: nothing to do, and Xs, vwork and var are not needed
    assert _var(lib, _off([0, 0, 0]), off, 3, ks, Xs=None, vwork=None, var=None) == 0
    # a chunk whose gemm grid would exceed 65535 tiles is rejected, unless the problems have fewer test points
    big = _off([4096])
    limit = 65535 // 64 * 128
    assert _var(lib, _off([limit + 1]), big, 1, _sums(1), chunk=limit + 1) == -1
    assert b"grid limit" in lib.tgp_last_error()
    assert lib.tgp_predict_var_batch_work_doubles(_ptr(_off([limit + 1])), _ptr(big), 1, limit + 1) == -1
    assert lib.tgp_predict_var_batch_work_doubles(_ptr(_off([limit])), _ptr(big), 1, limit + 1) == limit * 4096
    wd = lambda s, o, B, c: lib.tgp_predict_var_batch_work_doubles(_ptr(s), _ptr(o), B, c)
    assert wd(soff, off, 0, 4) == -1 and b"B must be >= 1" in lib.tgp_last_error()
    assert wd(None, off, 3, 4) == -1 and wd(soff, None, 3, 4) == -1 and wd(soff, off, 3, 0) == -1
    # sum_b min(M_b, chunk) ld_b
    assert wd(_off([5, 0, 7]), _off([9, 20, 31]), 3, 6) == 5 * 10 + 0 + 6 * 32


def test_loo_batch_rejects_bad_arguments_without_a_gpu():
    _, lib = _lib()
    off = _off([10, 20, 30])
    ks = _sums(3)
    cases = [
        (dict(B=0), b"B must be >= 1"),
        (dict(off=None), b"off"),
        (dict(off=_off([10, 0, 30])), b"off must be strictly increasing"),
        (dict(off=_off([10, 4097, 30])), b"TGP_BATCH_MAX_N"),
        (dict(ks=None), b"ks"),
    ]
    for kw, msg in cases:
        a = dict(off=off, B=3, ks=ks)
        a.update(kw)
        assert _loo(lib, a["off"], a["B"], a["ks"]) == -1, msg
        err = lib.tgp_last_error()
        assert err.startswith(b"tgp_loo_batch: invalid argument") and msg in err, (msg, err)
    for name in ("X", "y", "e2", "work", "alpha", "scratch", "mean", "var", "info"):
        assert _loo(lib, off, 3, ks, **{name: None}) == -1, name
        assert b"null pointer" in lib.tgp_last_error()
    assert _loo(lib, off, 3, ks, work=ctypes.c_void_p(24)) == -1 and b"work must be 16-byte" in lib.tgp_last_error()
    assert _loo(lib, off, 3, ks, scratch=ctypes.c_void_p(24)) == -1
    assert b"scratch must be 16-byte" in lib.tgp_last_error()


def test_var_batch_chunk_plan_covers_every_row_within_budget_and_grid():
    from treegp_b200 import backend

    rng = np.random.default_rng(3)
    for _ in range(200):
        B = int(rng.integers(1, 12))
        sizes = [int(n) for n in rng.integers(1, 4097, size=B)]
        ssizes = [int(m) for m in rng.integers(0, 5000, size=B)]
        budget = int(rng.integers(1 << 20, 1 << 31))
        for b0, b1 in backend.plan_batch_chunks(sizes, budget):
            s, m = sizes[b0:b1], ssizes[b0:b1]
            chunk = backend.var_batch_chunk(m, s, budget)
            assert 1 <= chunk <= max(1, max(m))
            assert chunk <= backend.var_batch_chunk_limit(s)
            # every launch's grid: gemm row tiles x column tiles, and the K build's row tiles
            eff = min(chunk, max(m))
            assert -(-eff // 128) * -(-max(s) // 64) <= 65535 and -(-eff // 64) <= 65535
            # the passes cover every row of every problem
            passes = -(-max(m) // chunk) if max(m) else 0
            assert all(passes * chunk >= mb for mb in m)
            ld = [(n + 1) & ~1 for n in s]
            v = 8 * sum(min(mb, chunk) * l for mb, l in zip(m, ld))
            factors = 8 * backend.batch_work_doubles(s)
            if chunk > 1:   # the largest chunk that fits: one more row per problem would not
                assert factors + v <= budget
                if chunk < min(max(m), backend.var_batch_chunk_limit(s)):
                    assert factors + 8 * sum(min(mb, chunk + 1) * l for mb, l in zip(m, ld)) > budget
    # the grid limit, not the budget, caps many rows on small problems
    assert backend.var_batch_chunk([10 ** 7], [64], 1 << 40) == 65535 * 64
    assert backend.var_batch_chunk([10 ** 7], [4096], 1 << 40) == 65535 // 64 * 128


def test_gp_batch_var_and_loo_reject_bad_input_before_device_work(monkeypatch):
    from treegp_b200 import GPInterpolationBatch, backend

    def no_device(*a, **k):
        raise AssertionError("device touched")

    for name in ("loglike_batch", "predict_mean_batch", "predict_var_batch", "loo_batch", "as_points", "to_device"):
        monkeypatch.setattr(backend, name, no_device)
    rng = np.random.default_rng(0)
    Xs = [rng.uniform(size=(n, 2)) for n in (30, 40)]
    ys = [rng.normal(size=30), rng.normal(size=40)]
    gp = GPInterpolationBatch(kernel="RBF(1.0)", optimizer="none")
    gp.initialize(Xs, ys)
    with pytest.raises(ValueError, match="one set of positions per problem"):
        gp.predict_var(Xs[:1])
    with pytest.raises(ValueError, match=r"problem 1: positions must have shape \(M, 2\)"):
        gp.predict_var([Xs[0], rng.uniform(size=5)])
    with pytest.raises(ValueError, match=r"problem 0: positions must have shape \(M, 2\)"):
        gp.predict_var([rng.uniform(size=(5, 1)), Xs[1]])
    # a kernel that is not finite is named before any device work
    gp.kernels[1] = gp.kernels[1].clone_with_theta(np.array([np.nan]))
    with pytest.raises(np.linalg.LinAlgError, match="problem 1: the kernel has non-finite"):
        gp.loo_predict()
    with pytest.raises(np.linalg.LinAlgError, match="problem 1: the kernel has non-finite"):
        gp.predict_var(Xs)
