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


# ------------------------------------------------------------------ device channel layout of the 16-bit precisions
MAX_NFB_16BIT = 64       # padded_width is defined up to 1024 channels: the bottleneck of nb_filters_base 64


def padded_width(c):
    """Channel width a c-channel tensor takes on the device in the 16-bit precisions: max(32, next power of two >= c).
    It is the smallest width that the tensor-core convolutions (multiples of 32), the first-layer conv (Cout in
    {8, 16, 32, 64}) and the single-launch BatchNorm kernels (a power of two <= 1024) all accept.  Powers of two from
    32 up map to themselves."""
    c = int(c)
    if not 1 <= c <= 1024:
        raise ValueError('no 16-bit device layout for %d channels (1 ... 1024)' % c)
    return max(32, 1 << (c - 1).bit_length())


class GraphSpec(object):
    """Arguments of the reference's ``unet()`` (unet_2d_summary.py:123-124).

    ``padded=True`` gives the device spec of the 16-bit precisions (see device_spec): the same graph with every tensor
    width c stored as padded_width(c) channels, so the concat input of a dec<l>a block is padded_width(up) +
    padded_width(skip) channels.  The network input (1 channel) and the head output (2 channels) keep their widths."""

    def __init__(self, nb_filters_base=32, prop_dropout_base=0.25, upsampling_or_transpose='transpose', padded=False):
        assert upsampling_or_transpose in ('transpose', 'upsampling')
        self.nfb = int(nb_filters_base)
        self.drp = float(prop_dropout_base)
        self.up_mode = upsampling_or_transpose
        self.padded = bool(padded)
        n, P = self.nfb, (padded_width if padded else int)
        b = [Block('enc0a', 'conv', 1, P(n), 0), Block('enc0b', 'conv', P(n), P(n), 0)]
        for lvl in (1, 2, 3):
            w = n << lvl
            b += [Block('enc%da' % lvl, 'conv', P(w // 2), P(w), lvl), Block('enc%db' % lvl, 'conv', P(w), P(w), lvl)]
        b += [Block('bota', 'conv', P(8 * n), P(16 * n), 4), Block('botb', 'conv', P(16 * n), P(16 * n), 4)]
        self.cat_split = OrderedDict()     # dec<l>a -> how many of its input channels come from the up path (the rest: skip)
        c = 16 * n
        for lvl in (3, 2, 1, 0):
            w = n << lvl
            if self.up_mode == 'transpose':
                b.append(Block('up%d' % lvl, 'up', P(c), P(w), lvl))
                up = P(w)
            else:
                up = P(c)
            self.cat_split['dec%da' % lvl] = up
            b += [Block('dec%da' % lvl, 'conv', up + P(w), P(w), lvl), Block('dec%db' % lvl, 'conv', P(w), P(w), lvl)]
            c = w
        b.append(Block('head', 'head', P(n), 2, 0))
        self.blocks = b
        self.by_name = OrderedDict((x.name, x) for x in b)

    def device_spec(self, precision):
        """The spec the engine allocates and launches with: padded for 'bf16' / 'fp16', this spec for the fp32 check
        mode, whose kernels take any width.  nb_filters_base 32 and 64 pad to themselves."""
        if precision == 'fp32' or self.padded:
            return self
        if not 1 <= self.nfb <= MAX_NFB_16BIT:
            raise ValueError("precision %r supports nb_filters_base 1 ... %d (got %d); use precision='fp32'"
                             % (precision, MAX_NFB_16BIT, self.nfb))
        return GraphSpec(self.nfb, self.drp, self.up_mode, padded=True)

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


def _channel_index(spec, dspec, name):
    """(device position of every input channel, of every output channel) of block ``name``: a concat input's up-path
    channels [0, up) stay in place, its skip channels [up, up + skip) move to [P(up), P(up) + skip)"""
    blk = spec.by_name[name]
    cin = np.arange(blk.cin)
    if name in spec.cat_split:
        up = spec.cat_split[name]
        cin = np.concatenate([cin[:up], dspec.cat_split[name] + np.arange(blk.cin - up)])
    return cin, np.arange(blk.cout)


def _index(spec, dspec, key):
    """index of the real entries of Keras array ``key`` inside its device array"""
    name, p = key.split('/')
    cin, cout = _channel_index(spec, dspec, name)
    if p != 'kernel':
        return cout
    if spec.by_name[name].kind == 'up':      # (2, 2, Cout, Cin)
        return slice(None), slice(None), cout[:, None], cin[None, :]
    return slice(None), slice(None), cin[:, None], cout[None, :]


def pack(spec, dspec, w):
    """Keras-shaped arrays of ``spec`` (any subset of its weight keys) -> arrays of the device spec ``dspec``.  Padded
    entries are 0 (kernel, bias, gamma, beta, moving_mean) or 1 (moving_var): a padded channel's convolution output is
    then exactly 0, its batch mean and variance are 0, and everything downstream of it, gradients included, stays 0."""
    if dspec is spec:
        return OrderedDict((k, np.asarray(a, dtype=np.float32)) for k, a in w.items())
    shapes, out = dspec.weight_shapes(), OrderedDict()
    for k, a in w.items():
        d = (np.ones if k.endswith('/moving_var') else np.zeros)(shapes[k], np.float32)
        d[_index(spec, dspec, k)] = a
        out[k] = d
    return out


def unpack(spec, dspec, w):
    """inverse of pack: device arrays -> Keras-shaped arrays of ``spec``"""
    if dspec is spec:
        return OrderedDict((k, np.asarray(a, dtype=np.float32)) for k, a in w.items())
    return OrderedDict((k, np.ascontiguousarray(np.asarray(a, dtype=np.float32)[_index(spec, dspec, k)]))
                       for k, a in w.items())


def _align4(n):
    return (n + 3) // 4 * 4


def flat_layout(spec):
    """The engine's flat parameter buffers: (OrderedDict key -> (trainable?, offset, shape), trainable floats,
    non-trainable floats).  Trainable arrays (kernel, bias, gamma, beta) share one buffer, the moving statistics
    another; every array starts at a multiple of 4 floats."""
    slots, off_t, off_n = OrderedDict(), 0, 0
    for blk in spec.blocks:
        for p, shp in blk.param_shapes().items():
            n = int(np.prod(shp))
            if p in TRAINABLE:
                slots['%s/%s' % (blk.name, p)] = (True, off_t, shp)
                off_t += _align4(n)
            else:
                slots['%s/%s' % (blk.name, p)] = (False, off_n, shp)
                off_n += _align4(n)
    return slots, off_t, off_n


def _convert_flat(src, dst, flat, fn):
    slots, n = flat_layout(src)[:2]
    flat = np.asarray(flat, dtype=np.float32)
    if flat.shape != (n,):
        raise ValueError('expected a flat trainable-parameter vector of %d floats, got shape %s' % (n, flat.shape))
    arrays = fn(OrderedDict((k, flat[off:off + int(np.prod(shp))].reshape(shp)) for k, (tr, off, shp) in slots.items() if tr))
    slots, n = flat_layout(dst)[:2]
    out = np.zeros(n, np.float32)
    for k, a in arrays.items():
        off = slots[k][1]
        out[off:off + a.size] = a.ravel()
    return out


def pack_flat(spec, dspec, flat):
    """a vector over the trainable parameters (Adam's m or v) in flat_layout(spec) -> the same in flat_layout(dspec)"""
    return _convert_flat(spec, dspec, flat, lambda w: pack(spec, dspec, w))


def unpack_flat(spec, dspec, flat):
    """inverse of pack_flat"""
    return _convert_flat(dspec, spec, flat, lambda w: unpack(spec, dspec, w))


# ------------------------------------------------------------------ overlap-tile inference for images larger than the window
MAX_TILE = 2048          # largest tile edge: a 2048^2 canvas is one tile; a batch holds at most 8 * MAX_TILE^2 pixels


def inference_bytes_per_pixel(spec, elem_bytes):
    """device bytes of the inference activation buffers per batch pixel for the device spec ``spec``: every block's
    output, the max-pooled encoder outputs and the upsampled tensors of the 'upsampling' graph at ``elem_bytes`` per
    value, plus the fp32 input, logit and probability"""
    b = 12.
    for blk in spec.blocks:
        if blk.kind == 'head':
            continue
        b += blk.cout * elem_bytes / 4. ** blk.level
        if blk.name.startswith('enc') and blk.name.endswith('b'):
            b += blk.cout * elem_bytes / 4. ** (blk.level + 1)
    if spec.up_mode == 'upsampling':
        b += sum(spec.cat_split['dec%da' % l] * elem_bytes / 4. ** l for l in range(4))
    return b


def tile_limits(spec, elem_bytes):
    """(batch pixels per tile group, largest tile edge) of predict_tiled for the device spec ``spec``: the activation
    bytes of 8 transforms of a MAX_TILE^2 tile at nb_filters_base 32 (29.4 GiB peak in fp16), which every narrower
    network keeps; a wider one gets proportionally fewer pixels and the largest multiple of 128 that still fits 8 of
    its tiles"""
    ref = GraphSpec(32, upsampling_or_transpose=spec.up_mode)
    px = 8 * MAX_TILE * MAX_TILE
    px = min(px, int(px * inference_bytes_per_pixel(ref, elem_bytes) // inference_bytes_per_pixel(spec, elem_bytes)))
    T = MAX_TILE
    while 8 * T * T > px and T > 512:
        T -= 128
    return px, T


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
