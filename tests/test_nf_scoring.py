"""Host side of the Neurofinder scoring: the shared float arithmetic (nf_scores_from_matches) gives exactly what the
formulas it replaced gave, and the validation boxes of fit, taken from the band's corners, equal the reference's np.where
boxes.  No GPU needed."""
import numpy as np
import pytest
from scipy import ndimage

from deepcalcium.datasets import nf
from deepcalcium.models.neurons.unet_2d_summary import UNet2DSummary


# ---- nf_centers / nf_shapes / nf_mask_metrics as they were before the float arithmetic moved into one helper
def _old_centers(a, b, threshold=5):
    inds = nf._match_regions(a, b, threshold)
    n = 0
    for ra, ib in zip(a, inds):
        if ib is not None and np.sqrt(((ra.mean(axis=0) - b[ib].mean(axis=0)) ** 2).sum()) < threshold:
            n += 1
    with np.errstate(divide='ignore', invalid='ignore'):
        return np.float64(n) / np.float64(len(a)), np.float64(n) / np.float64(len(b))


def _old_shapes(a, b, threshold=5):
    inds = nf._match_regions(a, b, threshold)
    rates = []
    for ra, ib in zip(a, inds):
        if ib is None:
            continue
        sa = set(map(tuple, ra.tolist()))
        nhit = float(sum(1 for xy in map(tuple, b[ib].tolist()) if xy in sa))
        rates.append((nhit / len(ra), nhit / len(b[ib])))
    if not rates:
        return 0.0, 0.0
    r = np.asarray(rates, dtype=np.float64).mean(axis=0)
    return float(r[0]), float(r[1])


def _old_mask_metrics(m, mp):
    mp = np.asarray(mp)
    if np.sum(mp.round()) == 0:
        return 0., 0., 0., 0., 0.
    a, b = nf._label_regions(m), nf._label_regions(mp)
    r, p = _old_centers(a, b)
    i, e = _old_shapes(a, b)
    with np.errstate(divide='ignore', invalid='ignore'):
        f1 = np.float64(2.) * (r * p) / (r + p)
    return (float(p), float(r), float(i), float(e), float(f1))


def _blobs(rng, shape, density):
    return (ndimage.gaussian_filter(rng.random(shape), 1.2) > 1 - density * 0.5 - 0.25).astype(np.uint8)


def _pairs(seed, n):
    rng = np.random.default_rng(seed)
    for t in range(n):
        H, W = (int(v) for v in rng.integers(1, 72, 2))
        m = _blobs(rng, (H, W), rng.random()) if t % 4 else (rng.random((H, W)) < rng.random()).astype(np.uint8)
        mp = np.roll(m, tuple(int(v) for v in rng.integers(-4, 5, 2)), (0, 1))
        if t % 5 == 0:
            mp = (rng.random((H, W)) < 0.2).astype(np.uint8)
        if t % 9 == 0:
            m = np.zeros_like(m)                   # no truth region: recall and F1 are NaN
        if t % 11 == 0:
            mp = np.zeros_like(mp)                 # empty prediction: the early exit
        yield m, mp


def test_metrics_equal_the_previous_formulas_on_random_masks():
    kinds = set()
    for m, mp in _pairs(1, 400):
        old, new = _old_mask_metrics(m, mp), nf.nf_mask_metrics(m, mp)
        assert np.array_equal(np.array(old), np.array(new), equal_nan=True), (old, new)
        kinds.add(('nan' if np.isnan(new).any() else 'finite', 'zero' if not mp.any() else 'pred'))
    assert {('nan', 'pred'), ('finite', 'pred'), ('finite', 'zero')} <= kinds


def test_centers_and_shapes_keep_their_values_and_types():
    for m, mp in _pairs(2, 120):
        a, b = nf._label_regions(m), nf._label_regions(mp)
        oc, nc = _old_centers(a, b), nf.nf_centers(a, b)
        assert all(type(v) is np.float64 for v in nc)
        assert np.array_equal(np.array(oc), np.array(nc), equal_nan=True)
        assert _old_shapes(a, b) == nf.nf_shapes(a, b)


def test_helper_from_a_matching():
    # na = 0 with predictions: recall 0 / 0 = NaN, precision 0, no shapes
    assert np.array_equal(nf.nf_scores_from_matches(0, 3, [], [], [4, 5, 6], []), (0., np.nan, 0., 0., np.nan),
                          equal_nan=True)
    # two truth regions, one matched to prediction 1 with 3 of its 4 pixels inside the 6-pixel prediction region
    p, r, i, e, f1 = nf.nf_scores_from_matches(2, 2, [-1, 1], [5, 4], [9, 6], [0, 3])
    assert (p, r, i, e) == (0.5, 0.5, 0.75, 0.5) and f1 == 0.5


@pytest.mark.parametrize('shape', [(512, 512), (600, 560), (37, 53), (53, 37), (2, 9), (1, 1), (128, 1)])
def test_validation_box_from_corners_equals_np_where(shape):
    H, W = shape
    fwd = [lambda x: x, np.fliplr, np.flipud, lambda x: np.rot90(x, 1), lambda x: np.rot90(x, 2),
           lambda x: np.rot90(x, 3)]
    bands = {(H - int(H * 0.25), H)} | ({(0, H), (1, H), (H // 3, H // 3 + 1)} if H > 1 else {(0, 1)})
    for y0, y1 in bands:
        if y1 <= y0:
            continue
        vm = np.zeros(shape, np.uint8)
        vm[y0:y1, :] = 1
        for k, f in enumerate(fwd):
            yy, xx = np.where(f(vm) == 1)
            assert UNet2DSummary._val_box(shape, y0, y1, k) == (min(yy), max(yy), min(xx), max(xx)), (shape, y0, y1, k)
            # the signed-stride view _validate scores as truth is f_k of the mask
            src = UNet2DSummary._VAL_SRC[k]
            img = np.arange(H * W).reshape(H, W)
            fi = f(img)
            a, b = np.meshgrid(np.arange(fi.shape[0]), np.arange(fi.shape[1]), indexing='ij')
            i, j = src(H, W, a, b)
            assert np.array_equal(img[i, j], fi)
    with pytest.raises(ValueError):
        UNet2DSummary._val_box(shape, H, H, 0)
