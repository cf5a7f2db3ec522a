"""GPU: the TwoD count with super-chunk forms (super pairs in one bin, or varying along one axis, booked by the super
kernel; the classification pass skips their blocks) against the pair-by-pair kernel.  Counts identical, sums to
summation order, in catalogues dense enough that both super forms occur."""
import numpy as np
import pytest

import test_gpu_pairbin_split as tps

pytestmark = pytest.mark.gpu


def _dense(seed, lens, weighted):
    """Hilbert-sorted uniform catalogues back to back, each at about one point per unit area."""
    from treegp_b200 import backend

    rng = np.random.default_rng(seed)
    xs, ys = [], []
    for n in lens:
        L = np.sqrt(n)
        x, y = rng.uniform(0, L, n), rng.uniform(0, L, n)
        order = backend.hilbert_order(backend.to_device(x), backend.to_device(y)).cpu().numpy()
        xs.append(x[order])
        ys.append(y[order])
    x, y = np.concatenate(xs), np.concatenate(ys)
    k = rng.normal(size=len(x))
    w = rng.uniform(0.5, 2.0, len(x)) if weighted else None
    return x, y, k, w, np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)


def _counted(x, y, k, w, off, mx, nb, **kw):
    from treegp_b200 import backend

    backend.pairbin_stats(reset=True)
    res = tps._count(x, y, k, w, off, mx, nb, **kw)
    return res, backend.pairbin_stats(reset=True)


@pytest.mark.parametrize("weighted", [False, True])
def test_super_forms_dense_catalogue(gpu_ready, weighted):
    """N = 2e5 in a 447 x 447 field, 7 x 7 bins at half the diagonal: most super pairs are booked whole or by rank
    queries per row."""
    x, y, k, w, off = _dense(3, [200_000], weighted)
    mx = np.sqrt(2.0) * np.sqrt(200_000) / 2.0
    res, st = _counted(x, y, k, w, off, mx, 7)
    witness, st0 = _counted(x, y, k, w, off, mx, 7, block_sums=0)
    assert st["super_closed_form"] > 0 and st["super_one_axis"] > 0
    assert st0["super_closed_form"] == 0 and st0["super_one_axis"] == 0
    tps._same(res, witness)


@pytest.mark.parametrize("weighted", [False, True])
def test_super_forms_batched_catalogues_three_ranks(gpu_ready, weighted):
    """Catalogues of unequal length, one shorter than a super-chunk and one with a short last super-chunk, dealt to 3
    ranks with a small record cap."""
    x, y, k, w, off = _dense(19, [40_000, 100, 30_011, 25_600], weighted)
    res, st = _counted(x, y, k, w, off, 141.0, 7, nranks=3, record_cap=4096)
    witness, _ = _counted(x, y, k, w, off, 141.0, 7, block_sums=0)
    assert st["super_closed_form"] > 0 and st["super_one_axis"] > 0
    tps._same(res, witness)


def test_super_forms_lattice_on_bin_edges(gpu_ready):
    """A 300 x 300 lattice of spacing 0.5 with 4 x 4 bins of width 32: displacements sit exactly on bin edges, where
    the mirrored bin of a pair is not the mirror image of its forward bin, inside super pairs with one varying axis."""
    g = np.arange(0, 300, dtype=np.float64) * 0.5
    X, Y = np.meshgrid(g, g)
    x, y = X.ravel(), Y.ravel()
    from treegp_b200 import backend

    order = backend.hilbert_order(backend.to_device(x), backend.to_device(y)).cpu().numpy()
    x, y = x[order], y[order]
    k = np.random.default_rng(11).normal(size=len(x))
    off = np.array([0, len(x)], dtype=np.int64)
    res, st = _counted(x, y, k, None, off, 64.0, 4)
    witness, _ = _counted(x, y, k, None, off, 64.0, 4, block_sums=0)
    assert st["super_one_axis"] > 0
    tps._same(res, witness)


def test_super_forms_small_max_sep(gpu_ready):
    """max_sep = L / 100: nearly every super pair is out of range, and its blocks are skipped."""
    x, y, k, w, off = _dense(23, [200_000], False)
    mx = np.sqrt(200_000) / 100.0
    res, _ = _counted(x, y, k, w, off, mx, 21)
    witness, _ = _counted(x, y, k, w, off, mx, 21, block_sums=0)
    assert witness[0].sum() > 0
    tps._same(res, witness)
