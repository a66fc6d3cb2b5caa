"""Host statement of the dropout keep mask, the specification every kernel that draws it is held to.

Restates csrc/elementwise.cuh (philox4x32_10, dropout_scale8) in numpy: element e of a flat NHWC tensor draws the 16-bit
uniform half-word (e % 8) of Philox4x32-10(counter = (e / 8 low word, e / 8 high word, layer, 0), key = (seed low word,
seed high word)) - the low half of each of the words x, y, z, w in turn, then its high half - and is kept when that
half-word is >= uint32(float32(p) * 65536).  Kept elements are multiplied by the fp32 value 1 / (1 - p), dropped ones
by 0.  The seed a kernel draws with is its host seed, XORed with the device seed when it is given one.
"""
from collections import OrderedDict

import numpy as np

_M0, _M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
_W0, _W1 = 0x9E3779B9, 0xBB67AE85
_LO = np.uint64(0xFFFFFFFF)
_32 = np.uint64(32)


def philox4x32_10(c0, c1, c2, c3, k0, k1):
    """Philox4x32-10 (Salmon et al. 2011) on arrays of counters (broadcast) -> four uint32 arrays x, y, z, w"""
    c0, c1, c2, c3 = (np.asarray(c, dtype=np.uint64) & _LO for c in (c0, c1, c2, c3))
    k0, k1 = int(k0) & 0xFFFFFFFF, int(k1) & 0xFFFFFFFF
    for _ in range(10):
        p0, p1 = _M0 * c0, _M1 * c2                      # exact: both factors < 2^32
        c0, c1, c2, c3 = (p1 >> _32) ^ c1 ^ np.uint64(k0), p1 & _LO, (p0 >> _32) ^ c3 ^ np.uint64(k1), p0 & _LO
        k0, k1 = (k0 + _W0) & 0xFFFFFFFF, (k1 + _W1) & 0xFFFFFFFF
    return tuple(c.astype(np.uint32) for c in (c0, c1, c2, c3))


def threshold(p):
    """the half-word an element must reach to be kept"""
    return int(np.float32(p) * np.float32(65536))


def keep_value(p):
    """what a kept element is multiplied by (fp32, as the kernels compute it)"""
    return np.float32(1) / (np.float32(1) - np.float32(p))


def uniforms16(seed, layer, n):
    """the 16-bit uniforms of elements 0 .. n-1 (uint32 array)"""
    seed = int(seed) & 0xFFFFFFFFFFFFFFFF
    g = np.arange((int(n) + 7) // 8, dtype=np.uint64)
    words = philox4x32_10(g & _LO, g >> _32, np.uint64(layer), np.uint64(0), seed & 0xFFFFFFFF, seed >> 32)
    halves = np.empty((g.size, 8), dtype=np.uint32)
    for i, w in enumerate(words):
        halves[:, 2 * i] = w & 0xFFFF
        halves[:, 2 * i + 1] = w >> 16
    return halves.reshape(-1)[:n]


_cache = OrderedDict()


def keep_scale(seed, layer, n, p):
    """fp32 keep scale of elements 0 .. n-1: 1 / (1 - p) where kept, 0 where dropped (the last few results are cached:
    the tests compare many kernels with the same mask)"""
    key = (int(seed) & 0xFFFFFFFFFFFFFFFF, int(layer), int(n), float(p))
    if key not in _cache:
        k = np.where(uniforms16(seed, layer, n) >= threshold(p), keep_value(p), np.float32(0))
        k.setflags(write=False)
        _cache[key] = k
        while len(_cache) > 8:
            _cache.popitem(last=False)
    return _cache[key]


def _tensor_geometry(eng, name):
    """(level, device channels, logical channels) of a dropped-out tensor of the engine's graph"""
    if name in eng.dspec.by_name:
        blk = eng.dspec.by_name[name]
        return blk.level, blk.cout, eng.spec.by_name[name].cout
    dec = 'dec%sa' % name[2:]                           # nearest-upsampled tensor: the up part of dec<l>a's concat input
    return int(name[2:]), eng.dspec.cat_split[dec], eng.spec.cat_split[dec]


def engine_keep_masks(eng, B, H, W, dropout=True, step_seed=None):
    """{tensor name: 0/1 keep mask [B, C, h, w]} of the training step an engine has just run on a B x H x W batch, in the
    form oracle.unet_forward(dropout_keep=) takes (None when the step ran without dropout).  step_seed: the step's device
    seed, by default read from the engine's step state (the step advances it before its kernels read it).  In the 16-bit
    modes the mask is drawn over the padded device width and cropped to the logical channels."""
    if not dropout:
        return None
    if step_seed is None:
        step_seed = int(eng.step_state[1].item())
    seed = (eng.dropout_seed_base() ^ step_seed) & 0xFFFFFFFFFFFFFFFF
    masks = OrderedDict()
    for name, (layer, p) in eng.dropout_layers().items():
        level, c_dev, c = _tensor_geometry(eng, name)
        h, w = H >> level, W >> level
        k = keep_scale(seed, layer, B * h * w * c_dev, p).reshape(B, h, w, c_dev)[..., :c]
        masks[name] = np.ascontiguousarray((k > 0).transpose(0, 3, 1, 2)).astype(np.float64)
    return masks
