"""CPU: batches of independent problems without a GPU -- argument validation of the batch entry points, the workspace
formula, the chunk planner, the lock-step L-BFGS-B driver against sequential scipy runs (with an injected numpy
objective), and the input validation of GPInterpolationBatch, all before any device work."""
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


def _loglike(lib, off, B, ks, X=P16, y=P16, e2=P16, work=P16, alpha=P16, out=P16, info=P16):
    o = None if off is None else ctypes.c_void_p(off.ctypes.data)
    return lib.tgp_loglike_batch(X, y, e2, o, B, ks, work, alpha, 0, out, info, None)


def test_batch_entries_reject_bad_arguments_without_a_gpu():
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
        assert _loglike(lib, kw["off"], kw["B"], kw["ks"]) == -1, msg
        err = lib.tgp_last_error()
        assert err.startswith(b"tgp_loglike_batch: invalid argument") and msg in err, (msg, err)
    bad = _sums(3)
    bad[1].term[0].family = 99
    assert _loglike(lib, off, 3, bad) == -1 and b"kernel sum descriptor" in lib.tgp_last_error()
    mixed = _sums(3)
    mixed[2] = _sums(1, ndim=1)[0]
    assert _loglike(lib, off, 3, mixed) == -1 and b"same ndim" in lib.tgp_last_error()
    for name in ("X", "y", "e2", "work", "alpha", "out", "info"):
        assert _loglike(lib, off, 3, ks, **{name: None}) == -1, name
        assert b"null pointer" in lib.tgp_last_error()
    assert _loglike(lib, off, 3, ks, work=ctypes.c_void_p(24)) == -1 and b"16-byte" in lib.tgp_last_error()
    # predict: soff may have empty problems but must start at 0 and not decrease
    soff = np.array([0, 5, 5, 9], dtype=np.int64)
    p = lambda s, o, B, k, **kw: lib.tgp_predict_mean_batch(kw.get("Xs", P16), ctypes.c_void_p(s.ctypes.data), P16,
                                                             ctypes.c_void_p(o.ctypes.data), B, k, P16,
                                                             kw.get("mean", P16), None)
    assert p(np.array([0, 5, 4, 9], dtype=np.int64), off, 3, ks) == -1 and b"soff must be non-decreasing" in lib.tgp_last_error()
    assert p(soff, _off([3, 0, 3]), 3, ks) == -1 and b"off must be strictly increasing" in lib.tgp_last_error()
    assert p(soff, off, 3, ks, mean=None) == -1 and b"null pointer" in lib.tgp_last_error()
    assert p(soff, off, 0, ks) == -1 and b"B must be >= 1" in lib.tgp_last_error()


def test_batch_work_doubles_formula():
    _cabi, lib = _lib()
    from treegp_b200 import backend

    rng = np.random.default_rng(3)
    for sizes in ([1], [1, 2, 3], [63, 64, 65, 511, 512, 513], list(rng.integers(1, 4097, size=40)), [4096] * 3):
        off = _off(sizes)
        n = np.asarray(sizes, dtype=np.int64)
        expect = int(np.sum((n + 1) * ((n + 1) // 2 * 2)))
        assert lib.tgp_batch_work_doubles(ctypes.c_void_p(off.ctypes.data), len(sizes)) == expect
        assert backend.batch_work_doubles(sizes) == expect
    assert lib.tgp_batch_work_doubles(ctypes.c_void_p(_off([3, 0]).ctypes.data), 2) == -1
    assert lib.tgp_batch_work_doubles(ctypes.c_void_p(_off([4097]).ctypes.data), 1) == -1


def test_plan_batch_chunks_covers_in_order_within_budget():
    from treegp_b200 import backend

    rng = np.random.default_rng(5)
    sizes = list(rng.integers(1, 4097, size=200))
    for budget in (1, 8 * 4097 * 4096, 50 << 20, 1 << 30, 1 << 40):
        chunks = backend.plan_batch_chunks(sizes, budget)
        assert chunks[0][0] == 0 and chunks[-1][1] == len(sizes)
        assert all(a < b for a, b in chunks) and all(chunks[i][1] == chunks[i + 1][0] for i in range(len(chunks) - 1))
        for a, b in chunks:
            need = 8 * backend.batch_work_doubles(sizes[a:b])
            assert need <= budget or b - a == 1      # a single problem larger than the budget gets a chunk of its own
    assert backend.plan_batch_chunks(sizes, 1) == [(b, b + 1) for b in range(len(sizes))]
    assert backend.plan_batch_chunks(sizes, 1 << 40) == [(0, len(sizes))]
    assert backend.plan_batch_chunks([], 1 << 30) == []


def _objectives():
    """Six problems: smooth bowls of different shapes (finishing in different rounds) and one that is always -inf."""
    def bowl(c, s):
        return lambda th: float(np.sum(s * (np.asarray(th) - c) ** 2) + np.sum(np.cos(3 * np.asarray(th))) * 0.1)

    fs = [bowl(np.array([0.3, -1.0]), np.array([1.0, 4.0])),
          bowl(np.array([2.0]), np.array([0.5])),
          bowl(np.array([-0.5, 0.5, 1.5]), np.array([3.0, 1.0, 0.2])),
          lambda th: np.inf,                                  # -logL = +inf everywhere (logL = -inf)
          bowl(np.array([1.0, 1.0]), np.array([10.0, 0.1])),
          bowl(np.array([0.0]), np.array([100.0]))]
    x0s = [np.array([1.0, 1.0]), np.array([0.0]), np.array([0.0, 0.0, 0.0]), np.array([0.5, 0.5]),
           np.array([-2.0, 3.0]), np.array([0.7])]
    return fs, x0s


def test_lockstep_matches_sequential_scipy_exactly():
    from treegp_b200.gp_batch import lockstep_minimize

    fs, x0s = _objectives()
    rounds = []

    def evaluate(indices, thetas):
        rounds.append(len(indices))
        return [fs[b](t) for b, t in zip(indices, thetas)]

    before = threading.active_count()
    got = lockstep_minimize(evaluate, x0s)
    assert threading.active_count() == before
    for b in range(len(fs)):
        ref = optimize.minimize(fs[b], x0s[b], method="L-BFGS-B")["x"]
        assert np.array_equal(got[b], ref), b
    assert len(set(rounds)) > 1                # problems finished in different rounds
    assert rounds[0] == len(fs)


def test_lockstep_joins_every_thread_when_the_evaluator_raises():
    from treegp_b200.gp_batch import lockstep_minimize

    fs, x0s = _objectives()
    calls = []

    def evaluate(indices, thetas):
        calls.append(1)
        if len(calls) == 4:
            raise KeyError("device failure")
        return [fs[b](t) for b, t in zip(indices, thetas)]

    before = threading.active_count()
    with pytest.raises(KeyError, match="device failure"):
        lockstep_minimize(evaluate, x0s)
    assert threading.active_count() == before


def test_gp_batch_rejects_bad_input_before_device_work(monkeypatch):
    from treegp_b200 import GPInterpolationBatch, backend

    def no_device(*a, **k):
        raise AssertionError("device touched")

    for name in ("loglike_batch", "predict_mean_batch", "as_points", "to_device"):
        monkeypatch.setattr(backend, name, no_device)
    rng = np.random.default_rng(0)
    Xs = [rng.uniform(size=(n, 2)) for n in (30, 40)]
    ys = [rng.normal(size=30), rng.normal(size=40)]
    with pytest.raises(ValueError, match="optimizer"):
        GPInterpolationBatch(kernel="RBF(1.0)", optimizer="bogus")
    with pytest.raises(TypeError):
        GPInterpolationBatch(kernel=3)
    gp = GPInterpolationBatch(kernel="RBF(1.0)", optimizer="none")
    with pytest.raises(ValueError, match="same, non-zero length"):
        gp.initialize(Xs, ys[:1])
    with pytest.raises(ValueError, match="same, non-zero length"):
        gp.initialize(Xs, ys, [np.ones(30)])
    with pytest.raises(ValueError, match="1-D"):
        gp.initialize(Xs, [ys[0], rng.normal(size=(40, 2))])
    with pytest.raises(ValueError, match="GPInterpolation"):
        gp.initialize([rng.uniform(size=(4097, 2))], [rng.normal(size=4097)])
    with pytest.raises(ValueError, match="same ndim"):
        gp.initialize([Xs[0], rng.uniform(size=(40, 1))], ys)
    with pytest.raises(ValueError, match="kernel strings"):
        GPInterpolationBatch(kernel=["RBF(1.0)"] * 3, optimizer="none").initialize(Xs, ys)
    gp.initialize(Xs, ys)
    with pytest.raises(ValueError, match="means only"):
        gp.predict(Xs, return_cov=True)
    assert len(gp.kernels) == 2 and gp.kernels[0] is not gp.kernels[1]
