"""GPU: TwoD super pairs with one varying axis decided per row point by the staged leaf kernel, against a column
super-chunk staged once for many of them, and the classification pass reading each super pair's status from the
bitmap the super kernel leaves behind.  Against the pair-by-pair kernel: counts identical, sums to summation order.
Every case checks which kernel decided the one-axis super pairs: all of them the leaf kernel when its staged form
runs, none of them when it does not (bins too many for its tables, or the 2 x 2 per-row form switched off)."""
import numpy as np
import pytest

import test_gpu_pairbin_split as tps
import test_gpu_pairbin_super as tsup

pytestmark = pytest.mark.gpu

SUPER_PAIR = 256 * 256   # pairs of one super pair in pairbin_stats


def _check(x, y, k, w, off, mx, nb, fast_paths=7, **kw):
    """Count with the block forms and with the witness; returns the path statistics and the one-axis super pairs
    that the leaf kernel decided."""
    from treegp_b200 import backend

    backend.pairbin_stats(reset=True)
    backend.pairbin_super_one_axis_rows(reset=True)
    backend.set_option("pairbin_fast_paths", fast_paths)
    try:
        res = tps._count(x, y, k, w, off, mx, nb, **kw)
    finally:
        backend.set_option("pairbin_fast_paths", 7)
    st = backend.pairbin_stats(reset=True)
    rows = backend.pairbin_super_one_axis_rows(reset=True)
    witness = tps._count(x, y, k, w, off, mx, nb, block_sums=0)
    assert backend.pairbin_super_one_axis_rows(reset=True) == 0
    tps._same(res, witness)
    return st, rows


def _staged(st, rows):
    assert rows > 0
    assert rows * SUPER_PAIR == st["super_one_axis"]


def _hilbert(x, y):
    from treegp_b200 import backend

    order = backend.hilbert_order(backend.to_device(x), backend.to_device(y)).cpu().numpy()
    return x[order], y[order]


@pytest.mark.parametrize("weighted", [False, True])
def test_one_axis_rows_lattice_on_bin_edges(gpu_ready, weighted):
    """A 300 x 300 lattice of spacing 0.5 with 4 x 4 bins of width 32: displacements sit exactly on bin edges inside
    one-axis super pairs, so the mirrored-bit check at the split fails for some row points and their columns are
    moved to the exact mirrored bin in global memory."""
    g = np.arange(0, 300, dtype=np.float64) * 0.5
    X, Y = np.meshgrid(g, g)
    x, y = _hilbert(X.ravel(), Y.ravel())
    rng = np.random.default_rng(101)
    k = rng.normal(size=len(x))
    w = rng.uniform(0.5, 2.0, len(x)) if weighted else None
    off = np.array([0, len(x)], dtype=np.int64)
    _staged(*_check(x, y, k, w, off, 64.0, 4))


@pytest.mark.parametrize("weighted", [False, True])
def test_one_axis_rows_tied_coordinates(gpu_ready, weighted):
    """Half the points on 60 vertical lines, the other half on 60 horizontal lines, 7 x 7 bins at half the diagonal
    (bins about four super-chunks wide): column super-chunks hold long runs of equal coordinates along the varying
    axis."""
    rng = np.random.default_rng(103)
    n = 120_000
    L = np.sqrt(n)
    lines = (np.arange(60) + 0.3141) * (L / 60)
    x, y = rng.uniform(0, L, n), rng.uniform(0, L, n)
    x[: n // 2] = rng.choice(lines, n // 2)
    y[n // 2:] = rng.choice(lines, n - n // 2)
    x, y = _hilbert(x, y)
    k = rng.normal(size=n)
    w = rng.uniform(0.5, 2.0, n) if weighted else None
    off = np.array([0, n], dtype=np.int64)
    _staged(*_check(x, y, k, w, off, np.sqrt(2.0) * L / 2.0, 7))


@pytest.mark.parametrize("weighted", [False, True])
def test_one_axis_rows_unequal_catalogues_three_ranks(gpu_ready, weighted):
    """Catalogues of unequal length, one shorter than a super-chunk and one with a short last super-chunk, dealt to 3
    ranks with a small record cap: every rank sweeps all statuses into its bitmap, books and lists only its own super
    pairs, and its classification pass runs many rounds against the bitmap."""
    x, y, k, w, off = tsup._dense(107, [600, 40_000, 100, 30_011, 25_600], weighted)
    _staged(*_check(x, y, k, w, off, 141.0, 7, nranks=3, record_cap=4096))


@pytest.mark.parametrize("weighted", [False, True])
def test_one_axis_rows_many_bins_stay_in_super_kernel(gpu_ready, weighted):
    """99 x 99 bins: the tables and the CTA histogram of the staged leaf kernel do not fit in shared memory, so the
    super kernel decides the one-axis super pairs itself."""
    rng = np.random.default_rng(109)
    n, L = 100_000, np.sqrt(1000.0)   # 100 points per unit area: super-chunks about 1.6 units wide, bins about 4
    x, y = _hilbert(rng.uniform(0, L, n), rng.uniform(0, L, n))
    k = rng.normal(size=n)
    w = rng.uniform(0.5, 2.0, n) if weighted else None
    off = np.array([0, n], dtype=np.int64)
    st, rows = _check(x, y, k, w, off, 200.0, 99)
    assert st["super_one_axis"] > 0 and rows == 0


def test_one_axis_rows_without_per_row_form(gpu_ready):
    """pairbin_fast_paths without bit 1: no staged leaf kernel, and the super kernel decides the one-axis super pairs
    itself."""
    x, y, k, w, off = tsup._dense(113, [200_000], False)
    st, rows = _check(x, y, k, w, off, np.sqrt(2.0) * np.sqrt(200_000) / 2.0, 21, fast_paths=5)
    assert st["super_one_axis"] > 0 and rows == 0
