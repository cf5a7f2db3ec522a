"""CPU: the batched log-likelihood gradient without a GPU -- argument validation of tgp_loglike_grad_batch and its
scratch size, the scratch formula against the host one, the chunk planner with scratch, and the lock-step L-BFGS-B
driver with analytic gradients against sequential scipy runs, all before any device work."""
import ctypes
import threading

import numpy as np
import pytest
from scipy import optimize

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


def _grad(lib, off, B, ks, X=P16, y=P16, e2=P16, work=P16, alpha=P16, out=P16, info=P16, scratch=P16):
    o = None if off is None else ctypes.c_void_p(off.ctypes.data)
    return lib.tgp_loglike_grad_batch(X, y, e2, o, B, ks, work, alpha, out, info, scratch, None)


def test_grad_batch_entries_reject_bad_arguments_without_a_gpu():
    _cabi, lib = _lib()
    off = _off([10, 20, 30])
    ks = _sums(3)
    cases = [
        (dict(off=off, B=0, ks=ks), b"B must be >= 1"),
        (dict(off=None, B=3, ks=ks), b"off"),
        (dict(off=_off([10, 0, 30]), B=3, ks=ks), b"off must be strictly increasing"),
        (dict(off=np.array([0, 10, 5, 40], dtype=np.int64), B=3, ks=ks), b"off must be strictly increasing"),
        (dict(off=np.array([1, 10, 20, 30], dtype=np.int64), B=3, ks=ks), b"off[0] must be 0"),
        (dict(off=_off([10, 4097, 30]), B=3, ks=ks), b"TGP_BATCH_MAX_N"),
        (dict(off=off, B=3, ks=None), b"ks"),
    ]
    for kw, msg in cases:
        assert _grad(lib, kw["off"], kw["B"], kw["ks"]) == -1, msg
        err = lib.tgp_last_error()
        assert err.startswith(b"tgp_loglike_grad_batch: invalid argument") and msg in err, (msg, err)
    bad = _sums(3)
    bad[1].term[0].family = 99
    assert _grad(lib, off, 3, bad) == -1 and b"kernel sum descriptor" in lib.tgp_last_error()
    mixed = _sums(3)
    mixed[2] = _sums(1, ndim=1)[0]
    assert _grad(lib, off, 3, mixed) == -1 and b"same ndim" in lib.tgp_last_error()
    for name in ("X", "y", "e2", "work", "alpha", "out", "info", "scratch"):
        assert _grad(lib, off, 3, ks, **{name: None}) == -1, name
        assert b"null pointer" in lib.tgp_last_error()
    assert _grad(lib, off, 3, ks, work=ctypes.c_void_p(24)) == -1 and b"work must be 16-byte" in lib.tgp_last_error()
    assert _grad(lib, off, 3, ks, scratch=ctypes.c_void_p(24)) == -1
    assert b"scratch must be 16-byte" in lib.tgp_last_error()
    # the scratch size rejects what the entry rejects
    wd = lambda o, B: lib.tgp_loglike_grad_batch_work_doubles(None if o is None else ctypes.c_void_p(o.ctypes.data), B)
    assert wd(off, 0) == -1 and b"B must be >= 1" in lib.tgp_last_error()
    assert wd(None, 3) == -1
    assert wd(_off([3, 0]), 2) == -1 and b"strictly increasing" in lib.tgp_last_error()
    assert wd(_off([4097]), 1) == -1 and b"TGP_BATCH_MAX_N" in lib.tgp_last_error()


def test_grad_batch_scratch_formula():
    _cabi, lib = _lib()
    from treegp_b200 import backend

    rng = np.random.default_rng(3)
    for sizes in ([1], [1, 2, 3], [63, 64, 65, 511, 512, 513], list(rng.integers(1, 4097, size=40)), [4096] * 3):
        off = _off(sizes)
        per = [lib.tgp_loglike_grad_sum_work_doubles(int(n), _cabi.MAX_TERMS) for n in sizes]
        assert all(p % 2 == 0 for p in per)   # every problem's block stays 16-byte aligned
        got = lib.tgp_loglike_grad_batch_work_doubles(ctypes.c_void_p(off.ctypes.data), len(sizes))
        assert got == sum(per) == backend.grad_batch_scratch_doubles(sizes)
    assert _cabi.GRAD_BATCH_OUT == 4 + 4 * _cabi.MAX_TERMS


def test_plan_batch_chunks_with_scratch_covers_in_order_within_budget():
    from treegp_b200 import backend

    rng = np.random.default_rng(5)
    sizes = list(rng.integers(1, 4097, size=200))
    need1 = lambda s: 8 * (backend.batch_work_doubles(s) + backend.grad_batch_scratch_doubles(s))
    for budget in (1, need1([4096]), 50 << 20, 1 << 30, 1 << 40):
        chunks = backend.plan_batch_chunks(sizes, budget, scratch=True)
        assert chunks[0][0] == 0 and chunks[-1][1] == len(sizes)
        assert all(a < b for a, b in chunks) and all(chunks[i][1] == chunks[i + 1][0] for i in range(len(chunks) - 1))
        for a, b in chunks:
            assert need1(sizes[a:b]) <= budget or b - a == 1
    # the scratch makes chunks smaller than the workspace alone
    assert len(backend.plan_batch_chunks(sizes, 1 << 30, scratch=True)) > len(backend.plan_batch_chunks(sizes, 1 << 30))
    assert backend.plan_batch_chunks(sizes, 1 << 40, scratch=True) == [(0, len(sizes))]
    assert backend.plan_batch_chunks([], 1 << 30, scratch=True) == []


def _objectives():
    """Six problems with analytic gradients: bowls of different shapes (finishing in different rounds) and one that is
    always -inf with a zero gradient."""
    def bowl(c, s):
        def f(th):
            th = np.asarray(th, dtype=float)
            return (float(np.sum(s * (th - c) ** 2) + 0.1 * np.sum(np.cos(3 * th))),
                    2 * s * (th - c) - 0.3 * np.sin(3 * th))
        return f

    fs = [bowl(np.array([0.3, -1.0]), np.array([1.0, 4.0])),
          bowl(np.array([2.0]), np.array([0.5])),
          bowl(np.array([-0.5, 0.5, 1.5]), np.array([3.0, 1.0, 0.2])),
          lambda th: (np.inf, np.zeros(len(th))),          # -logL = +inf everywhere (logL = -inf)
          bowl(np.array([1.0, 1.0]), np.array([10.0, 0.1])),
          bowl(np.array([0.0]), np.array([100.0]))]
    x0s = [np.array([1.0, 1.0]), np.array([0.0]), np.array([0.0, 0.0, 0.0]), np.array([0.5, 0.5]),
           np.array([-2.0, 3.0]), np.array([0.7])]
    return fs, x0s


def test_lockstep_with_gradients_matches_sequential_scipy_exactly():
    from treegp_b200.gp_batch import lockstep_minimize

    fs, x0s = _objectives()
    rounds = []

    def evaluate(indices, thetas):
        rounds.append(len(indices))
        return [fs[b](t) for b, t in zip(indices, thetas)]

    before = threading.active_count()
    got = lockstep_minimize(evaluate, x0s, jac=True)
    assert threading.active_count() == before
    for b in range(len(fs)):
        ref = optimize.minimize(fs[b], x0s[b], method="L-BFGS-B", jac=True)["x"]
        assert np.array_equal(got[b], ref), b
    assert len(set(rounds)) > 1                # problems finished in different rounds
    assert rounds[0] == len(fs)


def test_lockstep_with_gradients_joins_every_thread_when_the_evaluator_raises():
    from treegp_b200.gp_batch import lockstep_minimize

    fs, x0s = _objectives()
    calls = []

    def evaluate(indices, thetas):
        calls.append(1)
        if len(calls) == 3:
            raise KeyError("device failure")
        return [fs[b](t) for b, t in zip(indices, thetas)]

    before = threading.active_count()
    with pytest.raises(KeyError, match="device failure"):
        lockstep_minimize(evaluate, x0s, jac=True)
    assert threading.active_count() == before
