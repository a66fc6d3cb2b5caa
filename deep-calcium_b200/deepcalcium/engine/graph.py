"""Static description of the UNet2DS graph (deepcalcium/models/neurons/unet_2d_summary.py:123-224
of the reference) and the Keras-layout weight container.

Layer names are ours; the ORDER and per-layer array order reproduce Keras'
``model.get_weights()`` for the reference graph: per layer trainable then
non-trainable arrays, i.e. conv [kernel, bias], BN [gamma, beta, moving_mean,
moving_variance] -> 134 arrays for the default (transpose) graph.
"""
from collections import OrderedDict

import numpy as np

BN_EPS = 1e-3            # keras.layers.BatchNormalization default epsilon
BN_MOMENTUM_CONV = 0.99  # unet_2d_summary.py:165 (Keras default)
BN_MOMENTUM_UP = 0.5     # unet_2d_summary.py:157

PARAMS = {'conv': ('kernel', 'bias', 'gamma', 'beta', 'moving_mean', 'moving_var'),
          'up': ('kernel', 'bias', 'gamma', 'beta', 'moving_mean', 'moving_var'),
          'head': ('kernel', 'bias')}
TRAINABLE = ('kernel', 'bias', 'gamma', 'beta')


class Block(object):
    __slots__ = ('name', 'kind', 'cin', 'cout', 'level')

    def __init__(self, name, kind, cin, cout, level):
        self.name, self.kind, self.cin, self.cout, self.level = name, kind, cin, cout, level

    def kernel_shape(self):
        if self.kind == 'conv':
            return (3, 3, self.cin, self.cout)       # Keras Conv2D: HWIO
        if self.kind == 'up':
            return (2, 2, self.cout, self.cin)       # Keras Conv2DTranspose: (kh, kw, Cout, Cin)
        return (1, 1, self.cin, self.cout)

    def param_shapes(self):
        shp = OrderedDict(kernel=self.kernel_shape(), bias=(self.cout,))
        if self.kind != 'head':
            for p in ('gamma', 'beta', 'moving_mean', 'moving_var'):
                shp[p] = (self.cout,)
        return shp


class GraphSpec(object):
    """Arguments of the reference's ``unet()`` (unet_2d_summary.py:123-124)."""

    def __init__(self, nb_filters_base=32, prop_dropout_base=0.25, upsampling_or_transpose='transpose'):
        assert upsampling_or_transpose in ('transpose', 'upsampling')
        self.nfb = int(nb_filters_base)
        self.drp = float(prop_dropout_base)
        self.up_mode = upsampling_or_transpose
        n = self.nfb
        b = [Block('enc0a', 'conv', 1, n, 0), Block('enc0b', 'conv', n, n, 0)]
        for lvl in (1, 2, 3):
            w = n << lvl
            b += [Block('enc%da' % lvl, 'conv', w // 2, w, lvl), Block('enc%db' % lvl, 'conv', w, w, lvl)]
        b += [Block('bota', 'conv', 8 * n, 16 * n, 4), Block('botb', 'conv', 16 * n, 16 * n, 4)]
        c = 16 * n
        for lvl in (3, 2, 1, 0):
            w = n << lvl
            if self.up_mode == 'transpose':
                b.append(Block('up%d' % lvl, 'up', c, w, lvl))
                cat = 2 * w
            else:
                cat = c + w
            b += [Block('dec%da' % lvl, 'conv', cat, w, lvl), Block('dec%db' % lvl, 'conv', w, w, lvl)]
            c = w
        b.append(Block('head', 'head', n, 2, 0))
        self.blocks = b
        self.by_name = OrderedDict((x.name, x) for x in b)

    def dropout_after(self):
        """{tensor name: drop probability}, unet_2d_summary.py:179,185,191,198,204,210,216."""
        d = self.drp
        return OrderedDict([('enc1b', d), ('enc2b', 2 * d), ('enc3b', 2 * d),
                            ('up3', 2 * d), ('up2', 2 * d), ('up1', 2 * d), ('up0', d)])

    def weight_keys(self):
        return ['%s/%s' % (blk.name, p) for blk in self.blocks for p in PARAMS[blk.kind]]

    def weight_shapes(self):
        return OrderedDict(('%s/%s' % (blk.name, p), shp) for blk in self.blocks
                           for p, shp in blk.param_shapes().items())

    def flops_forward(self, H, W):
        """MAC*2 of conv + convT + head for one H x W image."""
        f = 0
        for blk in self.blocks:
            h, w = H >> blk.level, W >> blk.level
            if blk.kind == 'conv':
                f += 2 * h * w * 9 * blk.cin * blk.cout
            elif blk.kind == 'up':      # input is at level+1 resolution, 4 output pixels per input pixel
                f += 2 * (h // 2) * (w // 2) * 4 * blk.cin * blk.cout
            else:
                f += 2 * h * w * blk.cin * blk.cout
        return f

    def flops_train(self, H, W):
        """fwd + dgrad + wgrad GEMM flops actually executed per image (no dgrad for the first layer)."""
        f = 0
        for blk in self.blocks:
            h, w = H >> blk.level, W >> blk.level
            if blk.kind == 'conv':
                g = 2 * h * w * 9 * blk.cin * blk.cout
                f += g * (2 if blk.name == 'enc0a' else 3)
            elif blk.kind == 'up':
                f += 3 * 2 * (h // 2) * (w // 2) * 4 * blk.cin * blk.cout
            else:
                f += 3 * 2 * h * w * blk.cin * blk.cout
        return f


def _truncated_normal(rng, shape):
    """standard normal re-drawn where |z| > 2 (tf.truncated_normal, which Keras 2.0.6's VarianceScaling(distribution=
    'normal') - i.e. he_normal - samples from: the effective standard deviation is ~0.88 of the nominal one)"""
    z = rng.standard_normal(shape)
    bad = np.abs(z) > 2
    while bad.any():
        z[bad] = rng.standard_normal(int(bad.sum()))
        bad = np.abs(z) > 2
    return z


def he_normal_weights(spec, seed=None):
    """Fresh Keras-style initialisation: he_normal kernels (truncated normal, stddev sqrt(2 / fan_in) with fan_in =
    kh*kw*shape[-2], the Keras rule, which is 4*Cout for the transposed kernels), zero biases, BN gamma=1 beta=0
    mean=0 var=1."""
    rng = np.random.RandomState(seed)
    w = OrderedDict()
    for blk in spec.blocks:
        ks = blk.kernel_shape()
        fan_in = ks[0] * ks[1] * ks[2]
        if blk.kind == 'head':      # Keras default for Conv2D(2, 1): glorot_uniform
            limit = np.sqrt(6. / (ks[2] + ks[3]))
            w[blk.name + '/kernel'] = rng.uniform(-limit, limit, ks).astype(np.float32)
        else:
            w[blk.name + '/kernel'] = (_truncated_normal(rng, ks) * np.sqrt(2. / fan_in)).astype(np.float32)
        w[blk.name + '/bias'] = np.zeros(blk.cout, np.float32)
        if blk.kind != 'head':
            w[blk.name + '/gamma'] = np.ones(blk.cout, np.float32)
            w[blk.name + '/beta'] = np.zeros(blk.cout, np.float32)
            w[blk.name + '/moving_mean'] = np.zeros(blk.cout, np.float32)
            w[blk.name + '/moving_var'] = np.ones(blk.cout, np.float32)
    return w


def weights_to_list(spec, w):
    return [np.asarray(w[k]) for k in spec.weight_keys()]


def list_to_weights(spec, lst):
    keys = spec.weight_keys()
    if len(keys) != len(lst):
        raise ValueError('expected %d weight arrays, got %d' % (len(keys), len(lst)))
    shapes = spec.weight_shapes()
    out = OrderedDict()
    for k, a in zip(keys, lst):
        a = np.asarray(a, dtype=np.float32)
        if tuple(a.shape) != tuple(shapes[k]):
            raise ValueError('weight %s: expected shape %s, got %s' % (k, shapes[k], a.shape))
        out[k] = a
    return out


# ------------------------------------------------------------------ overlap-tile inference for images larger than the window
MAX_TILE = 2048          # largest tile edge: a 2048^2 canvas is one tile; a batch holds at most 8 * MAX_TILE^2 pixels


def receptive_reach(spec, block=16):
    """How far (in input pixels, on either side) the outputs of a ``block``-aligned run of ``block`` output pixels reach
    into the input: a 1-D dependency pass over the graph (conv 3x3 widens by one position at its level, max-pool and
    convT 2x2 / nearest upsampling are 2x index maps, the skip paths join by union).  Returns (left, right)."""
    def memo(fn):
        cache = {}

        def g(p):
            r = cache.get(p)
            if r is None:
                r = cache[p] = fn(p)
            return r
        return g

    # each tensor is a map: position at its level -> [lo, hi] interval of input positions it depends on; all maps are
    # non-decreasing in both ends, so a window's interval is (lo of its first position, hi of its last)
    def conv(f):
        return memo(lambda p: (f(p - 1)[0], f(p + 1)[1]))

    def pool(f):
        return memo(lambda p: (f(2 * p)[0], f(2 * p + 1)[1]))

    def up(f):
        return memo(lambda p: f(p // 2))

    def cat(f, g):
        return memo(lambda p: (min(f(p)[0], g(p)[0]), max(f(p)[1], g(p)[1])))

    t, skips = (lambda p: (p, p)), {}
    for blk in spec.blocks:
        if blk.kind == 'up':
            t = up(t)
        elif blk.kind == 'conv':
            if blk.name.startswith('dec') and blk.name.endswith('a'):
                t = cat(up(t) if spec.up_mode == 'upsampling' else t, skips[blk.level])
            t = conv(t)
            if blk.name.startswith('enc') and blk.name.endswith('b'):
                skips[blk.level] = t
                t = pool(t)
    return -t(0)[0], t(block - 1)[1] - (block - 1)


def tile_halo(spec):
    """h: the smallest multiple of 16 that covers the receptive reach.  A pixel at least h from every tile edge that is
    not a canvas edge gets the same prediction from the tile as from the whole canvas."""
    return -(-max(receptive_reach(spec)) // 16) * 16


def _round16(n):
    return -(-n // 16) * 16


def _plan_1d(C, T, h):
    """tile origins and ownership cuts along one canvas dimension of C pixels"""
    if C == T:
        return [0], []
    n = -(-(C - 2 * h) // (T - 2 * h))
    while True:
        # o_k = 16 * round(k (C - T) / (16 (n - 1))), halves rounded up
        o = [16 * ((2 * k * (C - T) + 16 * (n - 1)) // (32 * (n - 1))) for k in range(n)]
        if all(o[k + 1] - o[k] <= T - 2 * h for k in range(n - 1)):
            break
        n += 1
    return o, [(o[k] + o[k + 1] + T) // 2 for k in range(n - 1)]


class TilePlan(object):
    """Square T x T tiles over the canvas (the image reflect-padded at the bottom and right to C_h x C_w,
    C_d = max(T, roundup16(size_d))).  Tile (ty, tx) has its origin at (origins[0][ty], origins[1][tx]) and owns canvas
    rows [cuts[0][ty-1], cuts[0][ty]) and columns [cuts[1][tx-1], cuts[1][tx]) (up to the canvas edge at either end)."""
    __slots__ = ('shape', 'tile', 'halo', 'canvas', 'origins', 'cuts')

    def __init__(self, shape, tile, halo, canvas, origins, cuts):
        self.shape, self.tile, self.halo, self.canvas, self.origins, self.cuts = shape, tile, halo, canvas, origins, cuts

    @property
    def grid(self):
        return len(self.origins[0]), len(self.origins[1])

    @property
    def n_tiles(self):
        return len(self.origins[0]) * len(self.origins[1])

    def computed_pixels(self):
        return self.n_tiles * self.tile * self.tile

    def key(self):
        return (self.shape, self.tile, tuple(map(tuple, self.origins)), tuple(map(tuple, self.cuts)))


def plan_tiles(shape, halo, tile=None, max_tile=MAX_TILE):
    """Tile plan for an image of ``shape`` = (hs, ws).  Origins are multiples of 16 (the four max-pools see the canvas'
    phase), every tile lies inside the canvas (per-layer zero padding happens at the real canvas edge), and every pixel is
    owned by one tile and lies at least ``halo`` from each of its tile's edges that is not a canvas edge.
    ``tile=None`` picks T among the multiples of 128 in [512, max_tile] that minimise the computed pixels (ties: fewer
    tiles); an explicit ``tile`` must be a multiple of 16 greater than 2 * halo."""
    hs, ws = int(shape[0]), int(shape[1])
    if hs <= 0 or ws <= 0:
        raise ValueError('empty image %s' % (shape,))
    if tile is None:
        best = None
        for T in range(512, max_tile + 1, 128):
            p = plan_tiles((hs, ws), halo, T)
            if best is None or (p.computed_pixels(), p.n_tiles) < (best.computed_pixels(), best.n_tiles):
                best = p
        return best
    T = int(tile)
    if T % 16 or T <= 2 * halo:
        raise ValueError('tile %d must be a multiple of 16 greater than twice the halo (%d)' % (T, halo))
    canvas = (max(T, _round16(hs)), max(T, _round16(ws)))
    per_dim = [_plan_1d(C, T, halo) for C in canvas]
    return TilePlan((hs, ws), T, halo, canvas, [o for o, _ in per_dim], [c for _, c in per_dim])
