"""GPU: the TwoD leaf kernel deciding super pairs per row point against the column super-chunk staged in shared memory
(bisections on its sorted copies, the "both bits" quadrant from a dominance table built from the link between the two
sorted orders), against the pair-by-pair kernel.  Counts identical, sums to summation order; every case checks how many
super pairs took the per-row form."""
import numpy as np
import pytest

import test_gpu_pairbin_super as tsup
from test_gpu_pairbin_super_leaves import _check

pytestmark = pytest.mark.gpu


def _rows_check(x, y, k, w, off, mx, nb, **kw):
    from treegp_b200 import backend

    backend.pairbin_super_rows(reset=True)
    taken = _check(x, y, k, w, off, mx, nb, **kw)
    return taken, backend.pairbin_super_rows(reset=True)


def _hilbert(x, y):
    from treegp_b200 import backend

    order = backend.hilbert_order(backend.to_device(x), backend.to_device(y)).cpu().numpy()
    return x[order], y[order]


@pytest.mark.parametrize("weighted", [False, True])
def test_rows_tied_coordinates(gpu_ready, weighted):
    """Half the points on 60 vertical lines, the other half on 60 horizontal lines (N = 1.2e5 at about one point per
    unit area): super-chunks hold long runs of equal x or equal y, so the link between the x order and the y order
    as stored is what keeps the quadrant right."""
    rng = np.random.default_rng(61)
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
    taken, rows = _rows_check(x, y, k, w, off, np.sqrt(2.0) * L / 2.0, 21)
    assert 0 < rows <= taken


@pytest.mark.parametrize("weighted", [False, True])
def test_rows_and_blocks_in_one_count(gpu_ready, weighted):
    """A lattice of spacing 0.5 (displacements exactly on the edges of bins 32 wide, so the mirrored-bit check of its
    super pairs fails) beside a random field of the same density: in one count some super pairs go per row point and
    the others block by block."""
    rng = np.random.default_rng(67)
    g = np.arange(0, 200, dtype=np.float64) * 0.5
    X, Y = np.meshgrid(g, g)
    n2 = 40_000
    x = np.concatenate([X.ravel(), rng.uniform(0, 100, n2)])
    y = np.concatenate([Y.ravel(), rng.uniform(100, 200, n2)])
    x, y = _hilbert(x, y)
    k = rng.normal(size=len(x))
    w = rng.uniform(0.5, 2.0, len(x)) if weighted else None
    off = np.array([0, len(x)], dtype=np.int64)
    taken, rows = _rows_check(x, y, k, w, off, 64.0, 4)
    assert 0 < rows < taken


@pytest.mark.parametrize("weighted", [False, True])
def test_rows_unequal_catalogues_three_ranks(gpu_ready, weighted):
    """Catalogues of unequal length dealt to 3 ranks, among them two super-chunks only (one super pair) and one short
    of a super-chunk: each rank groups its own list, and groups of a single super pair make work items of one entry."""
    x, y, k, w, off = tsup._dense(71, [600, 40_000, 100, 30_011, 25_600], weighted)
    taken, rows = _rows_check(x, y, k, w, off, 141.0, 7, nranks=3)
    assert 0 < rows <= taken
