"""GPU: the TwoD count with the leaf kernel (super pairs that span at most 2 x 2 bins, the range edge counting as one,
decided block by block without records) against the pair-by-pair kernel.  Counts identical, sums to summation order;
every case checks that the leaf kernel took super pairs."""
import numpy as np
import pytest

import test_gpu_pairbin_split as tps
import test_gpu_pairbin_super as tsup

pytestmark = pytest.mark.gpu


def _check(x, y, k, w, off, mx, nb, **kw):
    from treegp_b200 import backend

    backend.pairbin_super_leaves(reset=True)
    res = tps._count(x, y, k, w, off, mx, nb, **kw)
    taken = backend.pairbin_super_leaves(reset=True)
    witness = tps._count(x, y, k, w, off, mx, nb, block_sums=0)
    assert backend.pairbin_super_leaves(reset=True) == 0
    assert taken > 0
    tps._same(res, witness)
    return taken


@pytest.mark.parametrize("weighted", [False, True])
def test_leaves_dense_catalogue(gpu_ready, weighted):
    """N = 2e5 at about one point per unit area, 21 x 21 bins at half the field diagonal: bins about twice as wide as
    a super-chunk, so many super pairs span exactly 2 x 2 bins."""
    x, y, k, w, off = tsup._dense(31, [200_000], weighted)
    _check(x, y, k, w, off, np.sqrt(2.0) * np.sqrt(200_000) / 2.0, 21)


@pytest.mark.parametrize("weighted", [False, True])
def test_leaves_batched_catalogues_three_ranks(gpu_ready, weighted):
    """Catalogues of unequal length, one shorter than a super-chunk and one with a short last super-chunk, dealt to 3
    ranks: each rank lists and decides its own super pairs."""
    x, y, k, w, off = tsup._dense(37, [40_000, 100, 30_011, 25_600], weighted)
    _check(x, y, k, w, off, 141.0, 7, nranks=3)


def test_leaves_lattice_on_bin_edges(gpu_ready):
    """A 300 x 300 lattice of spacing 0.5 with 4 x 4 bins of width 32: displacements sit exactly on bin edges inside
    super pairs of 2 x 2 bins, so the mirrored-bit checks fail and blocks go back to the pair-by-pair loop, whose
    mismatched pairs are moved to their exact mirrored bin."""
    from treegp_b200 import backend

    g = np.arange(0, 300, dtype=np.float64) * 0.5
    X, Y = np.meshgrid(g, g)
    x, y = X.ravel(), Y.ravel()
    order = backend.hilbert_order(backend.to_device(x), backend.to_device(y)).cpu().numpy()
    x, y = x[order], y[order]
    k = np.random.default_rng(41).normal(size=len(x))
    off = np.array([0, len(x)], dtype=np.int64)
    _check(x, y, k, None, off, 64.0, 4)


@pytest.mark.parametrize("weighted", [False, True])
def test_leaves_range_edge(gpu_ready, weighted):
    """max_sep = 30 with 3 x 3 bins of width 20 at N = 2e5 (super-chunks about 16 units wide): the range edge
    |dx| or |dy| = max_sep runs through many super pairs whose in-range part sits in one bin per axis."""
    x, y, k, w, off = tsup._dense(43, [200_000], weighted)
    _check(x, y, k, w, off, 30.0, 3)


def test_leaves_small_record_cap(gpu_ready):
    """The leaf kernel runs once before the rounds; a small record cap forces many rounds of the other blocks."""
    x, y, k, w, off = tsup._dense(47, [60_000], False)
    _check(x, y, k, w, off, np.sqrt(2.0) * np.sqrt(60_000) / 2.0, 21, record_cap=4096)
