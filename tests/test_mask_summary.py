"""The decomposition behind dcb_mask_summary, stated in numpy (tests/mask_corpus.py), equals the reference's sequential
_summarize_mask (oracle/masks.py) on a seeded corpus, and that corpus holds cases where the visiting order changes the
result.  No GPU needed."""
import numpy as np
import pytest

import mask_corpus as mc
from oracle.masks import summarize_mask_array


def _cases():
    rng = np.random.default_rng(17)
    cases = [mc.disks(rng, n, H, W) for n, H, W in ((1, 64, 64), (2, 40, 40), (300, 512, 512), (60, 97, 131))]
    m = mc.disks(rng, 40, 64, 48)
    m[3, 5, 5], m[4, 6, 6], m[5, 7, 7] = 2, -1, 127             # values other than 1 do not count
    cases.append(m)
    cases += [mc.checkerboard(40, 41), mc.diagonal_chain(30, 64, 64), np.zeros((0, 5, 7), np.int8),
              np.ones((2, 9, 9), np.int8)]
    return cases


@pytest.mark.parametrize('i', range(9))
def test_decomposition_equals_the_sequential_walk(i):
    m = _cases()[i]
    got, ncand, sizes = mc.decomposed(m)
    assert got.dtype == np.float64 and got.shape == m.shape[1:]
    assert np.array_equal(got, summarize_mask_array(m))
    assert int(sizes.sum()) == ncand


def test_order_corpus_is_order_sensitive_and_decomposes_exactly():
    cases = mc.order_corpus()
    differs = 0
    for m in cases:
        ref = summarize_mask_array(m)
        assert np.array_equal(mc.decomposed(m)[0], ref)
        differs += not np.array_equal(mc.raster_walk(m), ref)
    # the walk order is not a detail: raster order gives another mask on a good share of these cases
    assert differs >= 50, differs


def test_checkerboard_is_one_cluster_of_every_pixel():
    m = mc.checkerboard(64, 64)
    got, ncand, sizes = mc.decomposed(m)
    assert ncand == 64 * 64 and len(sizes) == 1 and np.array_equal(got, summarize_mask_array(m))
