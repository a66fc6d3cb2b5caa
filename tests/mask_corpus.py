"""Mask sets for the truth-mask summary tests (tests/test_mask_summary.py, tests/test_gpu_mask_summary.py) and a numpy
statement of the decomposition dcb_mask_summary computes: owners, candidate centres, clusters of the dilated candidate
map, and an ordered walk per cluster."""
import numpy as np
from scipy import ndimage

EIGHT = np.ones((3, 3), dtype=bool)


def disks(rng, n, H, W, rmin=4, rmax=9, dtype=np.int8):
    """n planes, each a disk of radius [rmin, rmax) at a uniform centre (clipped at the borders)"""
    m = np.zeros((n, H, W), dtype)
    for k in range(n):
        cy, cx, r = (int(v) for v in (rng.integers(0, H), rng.integers(0, W), rng.integers(rmin, rmax)))
        y0, x0 = max(cy - r, 0), max(cx - r, 0)
        yy, xx = np.mgrid[y0:min(cy + r + 1, H), x0:min(cx + r + 1, W)]
        m[k, y0:y0 + yy.shape[0], x0:x0 + yy.shape[1]] = (yy - cy) ** 2 + (xx - cx) ** 2 <= r * r
    return m


def order_corpus(seed=3, count=200):
    """small crowded cases (6 neurons of radius 3..5 in 24 x 24) in which the visiting order matters"""
    rng = np.random.default_rng(seed)
    return [disks(rng, 6, 24, 24, 3, 6) for _ in range(count)]


def owners(msks):
    """owner of every pixel: the plane that is == 1 there when exactly one is, else -1"""
    one = np.asarray(msks) == 1
    return np.where(one.sum(0) == 1, np.argmax(one, axis=0), -1) if len(one) else np.full(one.shape[1:], -1)


def _walk(own, alive, centres):
    H, W = own.shape
    for y, x in centres:
        y0, y1, x0, x1 = max(0, y - 1), min(H, y + 2), max(0, x - 1), min(W, x + 2)
        ow = own[y0:y1, x0:x1][alive[y0:y1, x0:x1]]
        if len(ow) and ow.min() != ow.max():
            alive[y0:y1, x0:x1] = False
    return alive


def decomposed(msks):
    """the summary as the device computes it -> (float64 [H, W], number of candidates, cluster sizes)"""
    own = owners(msks)
    H, W = own.shape
    alive = own >= 0
    pad = np.pad(own, 1, constant_values=-1)
    big = np.iinfo(np.int64).max
    mn, mx = np.full((H, W), big), np.full((H, W), -1)
    for dy in (0, 1, 2):
        for dx in (0, 1, 2):
            v = pad[dy:dy + H, dx:dx + W]
            mn = np.where(v >= 0, np.minimum(mn, v), mn)
            mx = np.maximum(mx, v)
    cand = alive & (mn < mx)
    lbl, nclus = ndimage.label(ndimage.binary_dilation(cand, EIGHT), structure=EIGHT)
    ys, xs = np.nonzero(cand)
    c = lbl[ys, xs]
    order = np.lexsort((xs, ys, own[ys, xs], c))            # by cluster, then (owner, y, x)
    sizes = np.bincount(c, minlength=nclus + 1)[1:]
    _walk(own, alive, zip(ys[order].tolist(), xs[order].tolist()))
    return alive.astype(np.float64), int(cand.sum()), sizes


def raster_walk(msks):
    """the same walk with every surviving pixel visited in raster order instead of (owner, y, x)"""
    own = owners(msks)
    ys, xs = np.nonzero(own >= 0)
    return _walk(own, own >= 0, zip(ys.tolist(), xs.tolist())).astype(np.float64)


def checkerboard(H, W):
    """two neurons interleaved as a checkerboard: every pixel is a candidate, all in one cluster"""
    ii, jj = np.meshgrid(np.arange(H), np.arange(W), indexing='ij')
    b = (ii + jj) % 2
    return np.stack([b == 0, b == 1]).astype(np.int8)


def diagonal_chain(n, H, W, size=6, step=2):
    """n square neurons along the main diagonal, each overlapping the next: one long cluster"""
    m = np.zeros((n, H, W), np.int8)
    for k in range(n):
        y, x = (k * step) % (H - size), (k * step) % (W - size)
        m[k, y:y + size, x:x + size] = 1
    return m
