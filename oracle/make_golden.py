"""Generate the committed known-answer fixtures under tests/golden/.

TEST INFRASTRUCTURE ONLY.  PARITY UNPINNED: the reference ships no golden vectors and cannot be
run here (Keras 2.0.6 / TF 1.2.1 absent), so these vectors come from the oracle restatement
itself (float64).  They pin the oracle against accidental change and give the GPU tests a
fixture that does not depend on recomputing the oracle.

To keep the fixture small, the U-Net weights are not stored: golden_weights() regenerates them
from the stored seed and checks them against the stored SHA-256 digest.  The gradient and the
updated weights of the largest tensor (botb/kernel, 3x3x64x64) are stored at a fixed seeded
sample of its entries, given by 'botb/kernel:index' (flat indices into the C-order array);
updated weights only for the tensors the tests check.

    python -m oracle.make_golden
"""
import hashlib
import os

import numpy as np
import torch

from . import (UNetSpec, init_weights, unet_forward, tta_predict, train_step, project_mean_max,
               summarize_series)

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'tests', 'golden')
WEIGHTS_SEED = 7535
SAMPLED = 'botb/kernel'
SAMPLE_SIZE = 2048


def weights_digest(w):
    h = hashlib.sha256()
    for k in sorted(w):
        a = np.ascontiguousarray(w[k])
        h.update(k.encode()); h.update(str(a.dtype).encode()); h.update(str(a.shape).encode()); h.update(a.tobytes())
    return h.hexdigest()


def golden_weights(z):
    """the nfb=4 weights the vectors of unet_nfb4_32.npz were computed from"""
    w = init_weights(UNetSpec(nb_filters_base=4), seed=int(z['weights_seed']))
    assert weights_digest(w) == str(z['weights_sha256']), 'oracle.init_weights no longer gives the golden weights'
    return w


def as_stored(z, key, a):
    """the full tensor ``a`` of parameter ``key`` reduced to the entries unet_nfb4_32.npz stores for it"""
    return np.asarray(a).ravel()[z[SAMPLED + ':index']] if key == SAMPLED else a


def main():
    os.makedirs(OUT, exist_ok=True)
    # --- projection: small int16-like movie
    rng = np.random.default_rng(7535)
    movie = (rng.random((37, 24, 40), dtype=np.float32) * 4096).astype(np.float32)
    mean, mx = project_mean_max(movie)
    np.savez_compressed(os.path.join(OUT, 'projection_small.npz'), movie=movie, mean=mean, max=mx,
                        summary=summarize_series(mean.astype(np.float16)))
    # --- tiny U-Net (nb_filters_base=4): forward, TTA, one training step per loss
    spec = UNetSpec(nb_filters_base=4)
    w = init_weights(spec, seed=WEIGHTS_SEED)
    x = np.random.default_rng(865).standard_normal((2, 32, 32)).astype(np.float32)
    y = (np.random.default_rng(866).random((2, 32, 32)) < 0.126).astype(np.uint8)
    fwd = unet_forward(w, x, spec, dtype=torch.float64)
    s = np.random.default_rng(3).standard_normal((27, 30)).astype(np.float32)
    mask, act = tta_predict(w, s, spec, window=32, dtype=torch.float64)
    idx = np.sort(np.random.default_rng(1).choice(w[SAMPLED].size, SAMPLE_SIZE, replace=False)).astype(np.int32)
    d = {'x': x, 'y': y, 'logit': fwd['logit'].numpy(), 'prob': fwd['prob'].numpy(), 's': s, 'tta_mask': mask,
         'tta_act': act, 'weights_seed': np.int64(WEIGHTS_SEED), 'weights_sha256': np.str_(weights_digest(w)),
         SAMPLED + ':index': idx}
    for loss in ('dice_loss', 'binary_crossentropy', 'dicesq_loss', 'weighted_binary_crossentropy'):
        L, nw, st, g, out = train_step(w, x, y, spec=spec, loss=loss)
        d['%s:loss' % loss] = np.float64(L)
        for k in ('enc0a/kernel', 'botb/kernel', 'up2/kernel', 'dec0b/gamma', 'head/kernel', 'head/bias'):
            d['%s:grad:%s' % (loss, k)] = as_stored(d, k, g[k])
        for k in ('botb/kernel', 'head/kernel'):
            d['%s:new:%s' % (loss, k)] = as_stored(d, k, nw[k])
        d['%s:new:enc0a/moving_mean' % loss] = nw['enc0a/moving_mean']
        d['%s:new:up1/moving_var' % loss] = nw['up1/moving_var']
    np.savez_compressed(os.path.join(OUT, 'unet_nfb4_32.npz'), **d)
    print('wrote', os.listdir(OUT))


if __name__ == '__main__':
    main()
