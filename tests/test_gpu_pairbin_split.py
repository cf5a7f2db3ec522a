"""GPU: the two-pass TwoD count (classification pass + pass over the recorded blocks) against the pair-by-pair
kernel.  Counts identical, sums to summation order, for what the other pair-binning tests do not reach: counts that
take many rounds of the record buffer, several catalogues dealt to three ranks, and a call without a work buffer."""
import ctypes

import numpy as np
import pytest

import test_gpu_pairbin as tpb

pytestmark = pytest.mark.gpu


def _catalogues(seed, lens, weighted):
    """Hilbert-sorted uniform catalogues back to back (dense enough that most blocks take the block forms)."""
    from treegp_b200 import backend

    rng = np.random.default_rng(seed)
    xs, ys = [], []
    for n in lens:
        x, y = rng.uniform(0, 400, n), rng.uniform(0, 400, n)
        order = backend.hilbert_order(backend.to_device(x), backend.to_device(y)).cpu().numpy()
        xs.append(x[order])
        ys.append(y[order])
    x, y = np.concatenate(xs), np.concatenate(ys)
    k = rng.normal(size=len(x))
    w = rng.uniform(0.5, 2.0, len(x)) if weighted else None
    return x, y, k, w, np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)


def _count(x, y, k, w, off, mx, nb, nranks=1, block_sums=1, record_cap=0):
    from treegp_b200 import backend

    backend.set_option("pairbin_block_sums", block_sums)
    backend.set_option("pairbin_record_cap", record_cap)
    try:
        return tpb._gpu_pairbin(x, y, k, w, 0.0, mx, nb, "TwoD", offsets=off, nranks=nranks)
    finally:
        backend.set_option("pairbin_block_sums", 1)
        backend.set_option("pairbin_record_cap", 0)


def _same(res, ref):
    np.testing.assert_array_equal(res[0], ref[0])
    np.testing.assert_allclose(res[1], ref[1], rtol=1e-12, atol=1e-12 * np.abs(ref[1]).max())
    np.testing.assert_allclose(res[2], ref[2], rtol=0, atol=tpb._kk_atol(ref[2], ref[1]))


@pytest.mark.parametrize("weighted", [False, True])
@pytest.mark.parametrize("mx", [280.0, 8.0])
def test_split_count_over_many_rounds(gpu_ready, weighted, mx):
    """The smallest record buffer (256 records: 8 items per round here) against one round and the witness.  At
    max_sep = 8 most items have no records."""
    from treegp_b200 import backend

    x, y, k, w, off = _catalogues(5, [40000], weighted)
    witness = _count(x, y, k, w, off, mx, 21, block_sums=0)
    backend.pairbin_stats(reset=True)
    one = _count(x, y, k, w, off, mx, 21)
    st1 = backend.pairbin_stats(reset=True)
    many = _count(x, y, k, w, off, mx, 21, record_cap=256)
    stm = backend.pairbin_stats(reset=True)
    if mx > 100:
        assert st1["closed_form"] > 0 and st1["one_axis_sorted"] > 0 and st1["two_axis_sorted"] > 0
    assert witness[0].sum() > 0
    assert stm == st1      # the rounds change when blocks are processed, not how
    _same(one, witness)
    _same(many, witness)


@pytest.mark.parametrize("weighted", [False, True])
def test_split_count_batched_catalogues_three_ranks(gpu_ready, weighted):
    """Catalogues of unequal length in one call, items dealt round-robin to 3 ranks, several rounds each."""
    x, y, k, w, off = _catalogues(9, [9000, 20011, 33, 14000], weighted)
    witness = _count(x, y, k, w, off, 280.0, 21, block_sums=0)
    one_rank = _count(x, y, k, w, off, 280.0, 21)
    three = _count(x, y, k, w, off, 280.0, 21, nranks=3, record_cap=4096)
    _same(one_rank, witness)
    _same(three, witness)


@pytest.mark.parametrize("weighted", [False, True])
def test_split_count_without_work_buffer(gpu_ready, weighted):
    """work == NULL: no pre-pass, so the pair-by-pair kernel; the same counts as with the work buffer."""
    import torch
    from treegp_b200 import _cabi, backend, binning

    x, y, k, w, off = _catalogues(13, [30000], weighted)
    nb, mx = 21, 280.0
    with_work = _count(x, y, k, w, off, mx, nb)
    dev = lambda a: backend.to_device(a)   # noqa: E731
    px, py, pk = dev(x), dev(y), dev(k)
    pw = None if w is None else dev(w)
    out = torch.zeros((3, 1, nb * nb), dtype=torch.float64, device=px.device)
    edges, coff = dev(binning.twod_thresholds(mx, nb)), backend.to_device(off, torch.int64)
    p = lambda t: ctypes.c_void_p(None if t is None else t.data_ptr())   # noqa: E731
    backend.pairbin_stats(reset=True)
    rc = _cabi.load().tgp_pairbin(p(px), p(py), p(pk), p(pw), p(coff), 1, len(x), _cabi.BIN_TWOD, p(edges), nb,
                                  0.0, mx, 0, 1, p(out[0]), p(out[1]), p(out[2]), p(None), p(None),
                                  ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert rc == 0
    st = backend.pairbin_stats(reset=True)
    assert st["closed_form"] == 0 and st["one_axis_sorted"] == 0 and st["two_axis_sorted"] == 0
    res = out.cpu().numpy()
    _same([res[0].view(np.int64), res[1], res[2]], with_work)


@pytest.mark.parametrize("weighted,nb", [(True, 40), (False, 64), (True, 90)])
def test_split_count_many_bins(gpu_ready, weighted, nb):
    """Bin counts whose warp histograms leave room for fewer than 8 warps per CTA in the classification pass."""
    x, y, k, w, off = _catalogues(17, [20000], weighted)
    _same(_count(x, y, k, w, off, 280.0, nb, record_cap=4096), _count(x, y, k, w, off, 280.0, nb, block_sums=0))
