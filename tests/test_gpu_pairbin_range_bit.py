"""GPU: the TwoD leaf kernel where the range edge is one of an axis' two slots (the range edge as a per-axis bit of the
super pair), and at bin counts near the shared-memory limit, against the pair-by-pair kernel.  Counts identical, sums to
summation order; every case checks that the leaf kernel took super pairs."""
import pytest

import test_gpu_pairbin_super as tsup
from test_gpu_pairbin_super_leaves import _check

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("weighted", [False, True])
def test_leaves_range_edge_both_axes_both_signs(gpu_ready, weighted):
    """max_sep = 10 with 2 x 2 bins against super-chunks about 16 units wide: the range edge crosses super pairs on
    both axes at once, at +max_sep and at -max_sep, so slots of either sign are out of range."""
    x, y, k, w, off = tsup._dense(53, [120_000], weighted)
    _check(x, y, k, w, off, 10.0, 2)


@pytest.mark.parametrize("weighted", [False, True])
def test_leaves_many_bins(gpu_ready, weighted):
    """99 x 99 bins of width 32 (max_sep = 1600 against a field 400 units wide): near the largest bin count for which
    the super kernel and the leaf kernel still run (the weighted warp histogram takes most of the shared memory)."""
    x, y, k, w, off = tsup._dense(59, [160_000], weighted)
    _check(x, y, k, w, off, 1600.0, 99)
