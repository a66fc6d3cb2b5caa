"""Losses, batch metrics and the test-time-augmentation table of the reference
(deepcalcium/utils/neurons.py:13-137), keeping its names.

In the reference these are Keras-backend graph functions; the names double as the keys of
``custom_objects`` (unet_2d_summary.py:329-331) and of the loss lookup (:372-377).  Here the
arithmetic of the loss, its gradient and the seven metrics runs inside the fused head kernels
(dcb_head_loss_fwd / dcb_head_loss_bwd); the functions below are host-side (numpy, float64)
evaluations of the same formulas for user code that calls them on arrays (e.g. scoring a
prediction), plus the id each name maps to in the C ABI.
"""
import numpy as np

from .._native import LOSS_IDS  # noqa: F401

K_EPSILON = 1e-7      # keras.backend.epsilon() in Keras 2.0.6


def _f(x):
    return np.asarray(x, dtype=np.float64)


def weighted_binary_crossentropy(yt, yp, weightpos=2., weightneg=1.):
    yt, yp = _f(yt), _f(yp)
    losspos = yt * np.log(yp + 1e-7)
    lossneg = (1 - yt) * np.log(1 - yp + 1e-7)
    return -1 * ((weightpos * losspos) + (weightneg * lossneg))


def binary_crossentropy(yt, yp):
    yt, yp = _f(yt), np.clip(_f(yp), K_EPSILON, 1 - K_EPSILON)
    return np.mean(-(yt * np.log(yp) + (1 - yt) * np.log(1 - yp)), axis=-1)


def prec(yt, yp):
    yt, yp = _f(yt), np.round(_f(yp))
    return np.sum(yp * yt) / (np.sum(yp) + K_EPSILON)


def reca(yt, yp):
    yt, yp = _f(yt), np.round(_f(yp))
    tp = np.sum(yp * yt)
    fn = np.sum(np.clip(yt - yp, 0, 1))
    return tp / (tp + fn + K_EPSILON)


def F1(yt, yp):
    p, r = prec(yt, yp), reca(yt, yp)
    return (2 * p * r) / (p + r + K_EPSILON)


def jacc(yt, yp):
    yt, yp = _f(yt), np.round(_f(yp))
    inter = np.sum(yt * yp)
    union = np.sum(yt) + np.sum(yp) - inter
    return inter / (union + 1e-7)


def jacc_loss(yt, yp):
    yt, yp = _f(yt), _f(yp)
    inter = np.sum(yt * yp)
    union = np.sum(yt) + np.sum(yp) - inter
    return 1 - inter / (union + 1e-7)


def dice(yt, yp):
    yt, yp = _f(yt), np.round(_f(yp))
    inter = np.sum(yt * yp)
    return (2. * inter) / (np.sum(yt) + np.sum(yp) + 1e-7)


def dice_loss(yt, yp):
    yt, yp = _f(yt), _f(yp)
    inter = np.sum(yt * yp)
    return 1 - (2. * inter) / (np.sum(yt) + np.sum(yp) + 1e-7)


def dicesq(yt, yp):
    yt, yp = _f(yt), _f(yp)
    nmr = 2 * np.sum(yt * yp)
    dnm = np.sum(yt ** 2) + np.sum(yp ** 2) + K_EPSILON
    return nmr / dnm


def dicesq_loss(yt, yp):
    return -1 * dicesq(yt, yp)


def posyt(yt, yp):
    yt = _f(yt)
    return np.sum(yt) / (yt.size + K_EPSILON)


def posyp(yt, yp):
    yp = _f(yp)
    return np.sum(np.round(yp)) / (yp.size + K_EPSILON)


# Order matters: it is the order of the transform index in dcb_tta_make_batch / dcb_tta_combine.
INVERTIBLE_2D_AUGMENTATIONS = [
    ('identity', lambda x: x, lambda x: x),
    ('vflip', lambda x: x[:, ::-1, ...], lambda x: x[:, ::-1, ...]),
    ('hflip', lambda x: x[:, :, ::-1], lambda x: x[:, :, ::-1]),
    ('rot90', lambda x: np.rot90(x, 1, axes=(1, 2)), lambda x: np.rot90(x, -1, axes=(1, 2))),
    ('rot180', lambda x: np.rot90(x, 2, axes=(1, 2)), lambda x: np.rot90(x, -2, axes=(1, 2))),
    ('rot270', lambda x: np.rot90(x, 3, axes=(1, 2)), lambda x: np.rot90(x, -3, axes=(1, 2))),
    ('rot90vflip', lambda x: np.rot90(x, 1, axes=(1, 2))[:, ::-1, ...],
     lambda x: np.rot90(x, 1, axes=(1, 2))[:, ::-1, ...]),
    ('rot90hflip', lambda x: np.rot90(x, 1, axes=(1, 2))[:, :, ::-1],
     lambda x: np.rot90(x, 1, axes=(1, 2))[:, :, ::-1]),
]


def tta_source_index(k, S, i, j):
    """Host mirror of the device index map in csrc/elementwise.cu (tta_src): source pixel of
    output (i,j) under transform k on an S x S image.  Tested against the table above."""
    return [(i, j), (S - 1 - i, j), (i, S - 1 - j), (j, S - 1 - i), (S - 1 - i, S - 1 - j),
            (S - 1 - j, i), (j, i), (S - 1 - j, S - 1 - i)][k]


def _reflect(i, n):
    """np.pad(mode='reflect') index map, extended to negative indices (reflect_index in csrc/elementwise.cu)"""
    if n == 1:
        return np.zeros_like(i)
    r = np.abs(i) % (2 * (n - 1))
    return np.where(r < n, r, 2 * (n - 1) - r)


def tile_make_batch_host(s, T, origins_y, origins_x, tile_first, n_tiles, first, count):
    """Host statement of dcb_tile_make_batch: [n_tiles * count, T, T] float32, the tiles tile_first.. of the plan (row-major
    over the origin grid) cut from the bottom / right reflect-padded canvas, each under transforms first..first+count-1."""
    s = np.asarray(s, np.float32)
    hs, ws = s.shape
    out = np.empty((n_tiles * count, T, T), np.float32)
    for lt in range(n_tiles):
        t = tile_first + lt
        y0, x0 = origins_y[t // len(origins_x)], origins_x[t % len(origins_x)]
        tile = s[np.ix_(_reflect(np.arange(y0, y0 + T), hs), _reflect(np.arange(x0, x0 + T), ws))][None]
        for kk in range(count):
            out[lt * count + kk] = INVERTIBLE_2D_AUGMENTATIONS[first + kk][1](tile)[0]
    return out


def tile_combine_host(probs, T, hs, ws, origins_y, origins_x, cuts_y, cuts_x, tile_first, n_tiles, n_aug, act=None):
    """Host statement of dcb_tile_combine: writes act [hs, ws] (float64) at the pixels owned by the group's tiles, the sum
    over the transforms in order of inv_k(p_k) / n_aug taken in the dtype of ``probs`` (float32 on the device).  Returns
    act; the mask is act > threshold."""
    act = np.zeros((hs, ws)) if act is None else act
    n_ty, n_tx = len(origins_y), len(origins_x)
    for lt in range(n_tiles):
        t = tile_first + lt
        ty, tx = t // n_tx, t % n_tx
        y0, x0 = origins_y[ty], origins_x[tx]
        p = probs[lt * n_aug:(lt + 1) * n_aug]
        acc = np.zeros((T, T))
        if n_aug == 1:
            acc += p[0]
        else:
            for k, (_, _, inv) in enumerate(INVERTIBLE_2D_AUGMENTATIONS):
                acc += inv(p[k:k + 1])[0] / n_aug
        r0, r1 = max(y0, cuts_y[ty - 1] if ty > 0 else 0), min(y0 + T, cuts_y[ty] if ty < n_ty - 1 else y0 + T, hs)
        c0, c1 = max(x0, cuts_x[tx - 1] if tx > 0 else 0), min(x0 + T, cuts_x[tx] if tx < n_tx - 1 else x0 + T, ws)
        if r0 < r1 and c0 < c1:
            act[r0:r1, c0:c1] = acc[r0 - y0:r1 - y0, c0 - x0:c1 - x0]
    return act


# ---------------------------------------------------------------------------------------------- outlined figures
_COLORS = {'red': (1., 0., 0.), 'blue': (0., 0., 1.), 'green': (0., 0.5, 0.), 'white': (1., 1., 1.), 'yellow': (1., 1., 0.)}


def mask_outlines(img, mask_arrs=(), colors=()):
    """utils/neurons.py:183-227 of the reference: the base image clipped at its 99th percentile and scaled to [0, 1], with
    the outline of every mask drawn in its colour, as a uint8 RGB array.  The reference strokes the mask through the
    un-vendored `regional` package; here the stroke is the mask's inner boundary (mask pixels with a 4-neighbour outside
    the mask), which is what `regional.one.mask(stroke=...)` draws up to its stroke width."""
    assert len(mask_arrs) == len(colors), 'One color per mask.'
    img = np.asarray(img, dtype=np.float32)
    img = np.clip(img, 0, np.percentile(img, 99))
    rng = float(np.max(img) - np.min(img))
    img = (img - np.min(img)) / (rng if rng > 0 else 1.0)
    rgb = np.repeat(img[:, :, None], 3, axis=2)
    oln = np.zeros_like(rgb)
    for m, c in zip(mask_arrs, colors):
        m = np.asarray(m) == 1
        if not m.any():
            continue
        p = np.pad(m, 1, mode='constant')
        inner = p[1:-1, 1:-1] & p[:-2, 1:-1] & p[2:, 1:-1] & p[1:-1, :-2] & p[1:-1, 2:]
        edge = m & ~inner
        col = _COLORS[c] if isinstance(c, str) else tuple(c)
        for k in range(3):
            oln[:, :, k][edge] = col[k]
    oln_msk = np.max(oln, axis=-1, keepdims=True)
    return (((oln * oln_msk) + rgb * (1 - oln_msk)) * 255).astype(np.uint8)
