"""Oracle: the UNet2DS graph, 8x TTA predict and one Keras-style training step.

TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).  PARITY UNPINNED.

Follows deepcalcium/models/neurons/unet_2d_summary.py:123-224 (graph),
:532-595 (predict / reflect pad / TTA / threshold) and the Keras 2.0.6 layer
semantics the graph inherits (not vendored in the reference; restated from the
pinned versions' documented behaviour):
  * Conv2D: HWIO kernel, bias, zero 'same' padding, cross-correlation.
  * Conv2DTranspose(2, strides=2): kernel (2,2,Cout,Cin),
    out[n,2i+a,2j+b,co] = sum_ci in[n,i,j,ci] * W[a,b,co,ci] + bias[co].
  * BatchNormalization(axis=-1, epsilon=1e-3): train = batch mean / biased
    variance over (N,H,W); moving <- moving*m + batch*(1-m); m=0.99 for conv
    blocks, 0.5 for up blocks (unet_2d_summary.py:157,165).
  * head: Conv2D(2, 1, softmax) then channel -1 (:221-222).
  * Adam in the Keras form (epsilon outside the bias correction).
torch (CPU) supplies conv arithmetic and autograd; nothing here uses torch's
BatchNorm / Adam defaults, which differ from Keras.
"""
from collections import OrderedDict
from dataclasses import dataclass

import numpy as np
import torch
import torch.nn.functional as F

from .losses import LOSSES, INVERTIBLE_2D_AUGMENTATIONS

BN_EPS = 1e-3


@dataclass(frozen=True)
class UNetSpec:
    """Arguments of ``unet()`` (unet_2d_summary.py:123-124)."""
    nb_filters_base: int = 32
    prop_dropout_base: float = 0.25
    upsampling_or_transpose: str = 'transpose'

    def blocks(self):
        """[(name, kind, cin, cout)] in layer-creation order; kind in
        {'conv','up','head'}.  Concat order is [upsampled, skip] (:200-218)."""
        n = self.nb_filters_base
        tr = self.upsampling_or_transpose == 'transpose'
        out = [('enc0a', 'conv', 1, n), ('enc0b', 'conv', n, n),
               ('enc1a', 'conv', n, 2 * n), ('enc1b', 'conv', 2 * n, 2 * n),
               ('enc2a', 'conv', 2 * n, 4 * n), ('enc2b', 'conv', 4 * n, 4 * n),
               ('enc3a', 'conv', 4 * n, 8 * n), ('enc3b', 'conv', 8 * n, 8 * n),
               ('bota', 'conv', 8 * n, 16 * n), ('botb', 'conv', 16 * n, 16 * n)]
        c = 16 * n
        for lvl, width in ((3, 8 * n), (2, 4 * n), (1, 2 * n), (0, n)):
            if tr:
                out.append(('up%d' % lvl, 'up', c, width))
                cat = 2 * width
            else:
                cat = c + width
            out.append(('dec%da' % lvl, 'conv', cat, width))
            out.append(('dec%db' % lvl, 'conv', width, width))
            c = width
        out.append(('head', 'head', n, 2))
        return out

    def dropout_after(self):
        """{tensor name: drop probability} (:179,185,191,198,204,210,216)."""
        d = self.prop_dropout_base
        return OrderedDict([('enc1b', d), ('enc2b', 2 * d), ('enc3b', 2 * d),
                            ('up3', 2 * d), ('up2', 2 * d), ('up1', 2 * d), ('up0', d)])


LAYER_ORDER = [b[0] for b in UNetSpec().blocks()]


def init_weights(spec=UNetSpec(), seed=7535, randomize_bn=True):
    """he_normal kernels, zero biases; BN stats optionally randomised so folding
    errors are visible (SURVEY.md section 8d).  Returns {name/param: float32}."""
    rng = np.random.default_rng(seed)
    w = OrderedDict()
    for name, kind, cin, cout in spec.blocks():
        if kind == 'conv':
            w[name + '/kernel'] = (rng.standard_normal((3, 3, cin, cout)) * np.sqrt(2. / (9 * cin))).astype(np.float32)
        elif kind == 'up':
            w[name + '/kernel'] = (rng.standard_normal((2, 2, cout, cin)) * np.sqrt(2. / (4 * cout))).astype(np.float32)
        else:
            w[name + '/kernel'] = (rng.standard_normal((1, 1, cin, cout)) * np.sqrt(2. / cin)).astype(np.float32)
        w[name + '/bias'] = (0.05 * rng.standard_normal(cout)).astype(np.float32) if randomize_bn \
            else np.zeros(cout, np.float32)
        if kind != 'head':
            if randomize_bn:
                w[name + '/gamma'] = (1 + 0.1 * rng.standard_normal(cout)).astype(np.float32)
                w[name + '/beta'] = (0.1 * rng.standard_normal(cout)).astype(np.float32)
                w[name + '/moving_mean'] = (0.1 * rng.standard_normal(cout)).astype(np.float32)
                w[name + '/moving_var'] = rng.uniform(0.5, 1.5, cout).astype(np.float32)
            else:
                w[name + '/gamma'] = np.ones(cout, np.float32)
                w[name + '/beta'] = np.zeros(cout, np.float32)
                w[name + '/moving_mean'] = np.zeros(cout, np.float32)
                w[name + '/moving_var'] = np.ones(cout, np.float32)
    return w


_PARAMS = {'conv': ['kernel', 'bias', 'gamma', 'beta', 'moving_mean', 'moving_var'],
           'up': ['kernel', 'bias', 'gamma', 'beta', 'moving_mean', 'moving_var'],
           'head': ['kernel', 'bias']}
TRAINABLE = ('kernel', 'bias', 'gamma', 'beta')


def weights_to_keras_list(w, spec=UNetSpec()):
    """``model.get_weights()`` order: per layer, trainable then non-trainable
    (conv k,b ; BN gamma,beta,mean,var) -> 134 arrays for the default graph."""
    return [w['%s/%s' % (name, p)] for name, kind, _, _ in spec.blocks() for p in _PARAMS[kind]]


def keras_list_to_weights(lst, spec=UNetSpec()):
    keys = ['%s/%s' % (name, p) for name, kind, _, _ in spec.blocks() for p in _PARAMS[kind]]
    assert len(keys) == len(lst)
    return OrderedDict(zip(keys, lst))


class _RoundBF16(torch.autograd.Function):
    """Round-to-nearest-even to bfloat16 with a straight-through gradient: models the bf16 storage of
    weights / raw conv outputs / activations in the tensor-core mode (accumulation stays exact)."""

    @staticmethod
    def forward(ctx, t):
        return t.to(torch.bfloat16).to(t.dtype)

    @staticmethod
    def backward(ctx, g):
        return g


def _conv3x3(x, k, b):
    return F.conv2d(x, k.permute(3, 2, 0, 1), b, padding=1)


def _convT2x2(x, k, b):
    # Keras kernel (2,2,Cout,Cin) -> torch conv_transpose2d weight (Cin,Cout,kh,kw)
    return F.conv_transpose2d(x, k.permute(3, 2, 0, 1), b, stride=2)


def _bn(x, g, be, mm, mv, training, stats_out, name):
    if training:
        mean = x.mean(dim=(0, 2, 3))
        var = ((x - mean[None, :, None, None]) ** 2).mean(dim=(0, 2, 3))
        stats_out[name] = (mean.detach(), var.detach())
    else:
        mean, var = mm, mv
    inv = torch.rsqrt(var + BN_EPS) * g
    return (x - mean[None, :, None, None]) * inv[None, :, None, None] + be[None, :, None, None]


def unet_forward(w, x, spec=UNetSpec(), training=False, dropout_keep=None, dtype=torch.float64,
                 return_intermediates=False, requires_grad=False, emulate_bf16=False, relu_gate=None):
    """Forward pass.  ``x``: [N,H,W] array.  Returns dict with
      'logit' = z1 - z0 (so prob = sigmoid(logit) = softmax(z)[..., -1]),
      'prob', and (training) 'bn_stats' {layer: (batch_mean, batch_var)}.
    ``dropout_keep``: {tensor name: 0/1 keep mask [N,C,H,W]} or None (= dropout
    off, the parity configuration).  With ``requires_grad`` the returned
    'params' dict holds leaf tensors for autograd.
    ``emulate_bf16``: round to bfloat16 exactly where the GPU's tensor-core mode stores bf16 - the
    kernels of every layer with Cin > 1, each raw conv output (after the bias) and each activation
    (after BN/ReLU/dropout) - keeping all arithmetic in ``dtype``.  This is the reference the bf16
    training path is compared with: the fp64 gradient of this randomly initialised dice-loss network is
    ill-conditioned w.r.t. 2^-9 perturbations of the activations (tens of percent), so only a
    reference with the same storage rounding isolates implementation errors.
    ``relu_gate``: {block name: 0/1 array [N,C,H,W]} - the block's ReLU keeps exactly the gated elements instead of
    deciding by the sign of its own pre-activation.  A pre-activation within a rounding error of 0 has no sign that
    every correct evaluation agrees on; a test can take those decisions from the implementation it checks.
    """
    rb = _RoundBF16.apply if emulate_bf16 else (lambda t: t)
    tw = OrderedDict((k, torch.tensor(np.asarray(v), dtype=dtype, requires_grad=(
        requires_grad and k.rsplit('/', 1)[1] in TRAINABLE))) for k, v in w.items())
    t = torch.as_tensor(np.ascontiguousarray(x), dtype=dtype)[:, None]   # NCHW, Cin=1 (:169-170)
    drops = spec.dropout_after()
    inter, stats = OrderedDict(), OrderedDict()

    def block(name, t):
        kind = 'up' if name.startswith('up') else 'conv'
        k = tw[name + '/kernel']
        if k.shape[2] > 1:          # the Cin = 1 first layer reads fp32 weights on the GPU as well
            k = rb(k)
        if kind == 'conv':
            t = _conv3x3(t, k, tw[name + '/bias'])
        else:
            t = _convT2x2(t, k, tw[name + '/bias'])
        if training:                # the raw output is only materialised (in bf16) for batch-stat BN
            t = rb(t)
        if return_intermediates:
            inter[name + '/raw'] = t
        t = _bn(t, tw[name + '/gamma'], tw[name + '/beta'], tw[name + '/moving_mean'],
                tw[name + '/moving_var'], training, stats, name)
        if relu_gate is not None and name in relu_gate:
            t = t * torch.as_tensor(relu_gate[name], dtype=dtype)
        else:
            t = torch.relu(t)
        if name not in drops or not (training and dropout_keep is not None):
            t = rb(t)
        if return_intermediates:
            inter[name] = t
        return t

    def drop(name, t):
        if training and dropout_keep is not None and name in dropout_keep:
            keep = 1. - drops[name]
            t = t * torch.as_tensor(dropout_keep[name], dtype=dtype) / keep
        return rb(t)                # activations are stored after ReLU (+ dropout)

    def up(lvl, t):
        if spec.upsampling_or_transpose == 'transpose':
            return drop('up%d' % lvl, block('up%d' % lvl, t))
        t = t.repeat_interleave(2, dim=2).repeat_interleave(2, dim=3)   # UpSampling2D (:160-161)
        return drop('up%d' % lvl, t)

    t = block('enc0b', block('enc0a', t)); s0 = t
    t = F.max_pool2d(t, 2)
    t = drop('enc1b', block('enc1b', block('enc1a', t))); s1 = t
    t = F.max_pool2d(t, 2)
    t = drop('enc2b', block('enc2b', block('enc2a', t))); s2 = t
    t = F.max_pool2d(t, 2)
    t = drop('enc3b', block('enc3b', block('enc3a', t))); s3 = t
    t = F.max_pool2d(t, 2)
    t = block('botb', block('bota', t))
    for lvl, skip in ((3, s3), (2, s2), (1, s1), (0, s0)):
        t = torch.cat([up(lvl, t), skip], dim=1)
        t = block('dec%db' % lvl, block('dec%da' % lvl, t))
    z = F.conv2d(t, tw['head/kernel'].permute(3, 2, 0, 1), tw['head/bias'])
    prob = torch.softmax(z, dim=1)[:, -1]
    out = {'logit': z[:, 1] - z[:, 0], 'prob': prob, 'bn_stats': stats, 'params': tw}
    if return_intermediates:
        out['intermediates'] = inter
    return out


def reflect_pad(x, hw=512, ww=512):
    """unet_2d_summary.py:569-571."""
    return np.pad(x, ((0, hw - x.shape[0]), (0, ww - x.shape[1])), mode='reflect')


def tta_predict(w, s, spec=UNetSpec(), augmentation=True, threshold=0.5, window=512, dtype=torch.float32):
    """unet_2d_summary.py:578-595 for one summary image ``s`` [hs,ws].
    Returns (mask uint8 [hs,ws], averaged activation float64 [hs,ws])."""
    hs, ws = s.shape
    s_batch = reflect_pad(s, window, window)[np.newaxis, :, :]

    def predict(xb):
        with torch.no_grad():
            return unet_forward(w, np.ascontiguousarray(xb), spec, dtype=dtype)['prob'].to(torch.float32).numpy()

    if augmentation:
        mp = np.zeros(s.shape)
        for _, aug, inv in INVERTIBLE_2D_AUGMENTATIONS:
            mpaug = predict(aug(s_batch))
            mp += inv(mpaug)[0, :hs, :ws] / len(INVERTIBLE_2D_AUGMENTATIONS)
    else:
        mp = predict(s_batch)[0, :hs, :ws]
    return (mp > threshold).astype(np.uint8), np.asarray(mp, dtype=np.float64)


def keras_adam_update(p, g, m, v, iteration, lr=0.002, beta_1=0.9, beta_2=0.999, epsilon=1e-8):
    """keras.optimizers.Adam.get_updates (Keras 2.0.6), numpy float64."""
    t = iteration + 1
    lr_t = lr * (np.sqrt(1. - beta_2 ** t) / (1. - beta_1 ** t))
    m_t = beta_1 * m + (1. - beta_1) * g
    v_t = beta_2 * v + (1. - beta_2) * np.square(g)
    p_t = p - lr_t * m_t / (np.sqrt(v_t) + epsilon)
    return p_t, m_t, v_t


def train_step(w, x, y, opt_state=None, spec=UNetSpec(), loss='dice_loss', lr=0.002,
               dropout_keep=None, dtype=torch.float64, emulate_bf16=False, relu_gate=None):
    """One ``train_on_batch``: forward with batch-stat BN, loss, autograd,
    Keras-Adam on the trainable tensors, momentum update of the BN moving stats.
    Returns (loss, new_weights, new_opt_state, grads, forward_out)."""
    out = unet_forward(w, x, spec, training=True, dropout_keep=dropout_keep, dtype=dtype, requires_grad=True,
                       emulate_bf16=emulate_bf16, relu_gate=relu_gate)
    yt = torch.as_tensor(np.asarray(y), dtype=dtype)
    L = LOSSES[loss](yt, out['prob'])
    params = {k: t for k, t in out['params'].items() if t.requires_grad}
    grads = torch.autograd.grad(L, list(params.values()), allow_unused=True)
    grads = {k: (np.zeros_like(np.asarray(w[k]), dtype=np.float64) if g is None else g.numpy().astype(np.float64))
             for k, g in zip(params.keys(), grads)}
    if opt_state is None:
        opt_state = {'iteration': 0, 'm': {k: np.zeros_like(g) for k, g in grads.items()},
                     'v': {k: np.zeros_like(g) for k, g in grads.items()}}
    new_w = OrderedDict((k, np.asarray(v).copy()) for k, v in w.items())
    new_state = {'iteration': opt_state['iteration'] + 1, 'm': {}, 'v': {}}
    for k, g in grads.items():
        p, m, v = keras_adam_update(np.asarray(w[k], np.float64), g, opt_state['m'][k], opt_state['v'][k],
                                    opt_state['iteration'], lr=lr)
        new_w[k] = p.astype(np.float32)
        new_state['m'][k], new_state['v'][k] = m, v
    for name, (mean, var) in out['bn_stats'].items():
        mom = 0.5 if name.startswith('up') else 0.99
        new_w[name + '/moving_mean'] = (np.asarray(w[name + '/moving_mean'], np.float64) * mom
                                        + mean.numpy() * (1 - mom)).astype(np.float32)
        new_w[name + '/moving_var'] = (np.asarray(w[name + '/moving_var'], np.float64) * mom
                                       + var.numpy() * (1 - mom)).astype(np.float32)
    return float(L.detach()), new_w, new_state, grads, out
