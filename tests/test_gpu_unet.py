"""End-to-end parity of the UNet2DS path on the GPU against the CPU oracle:
forward logits (fp32 check mode 1e-4, bf16 1e-2 class), 8x TTA masks (<= 0.1 % disagreement at
512^2), one training step (loss, gradients, updated weights, BN moving statistics), and the
reference-facing UNet2DSummary / unet() surface."""
import os

import numpy as np
import pytest
import torch

import oracle
from oracle.make_golden import as_stored, golden_weights

pytestmark = pytest.mark.gpu


def _engine(nfb, precision, w, **kw):
    from deepcalcium.engine.graph import GraphSpec
    from deepcalcium.engine.unet_engine import UNetEngine
    eng = UNetEngine(GraphSpec(nfb), precision=precision, **kw)
    eng.set_weights_dict(w)
    return eng


def test_golden_forward_fp32_check_mode(cuda, golden_dir):
    z = np.load(golden_dir + '/unet_nfb4_32.npz')
    w = golden_weights(z)
    eng = _engine(4, 'fp32', w)
    prob, logit = eng.infer(torch.from_numpy(z['x']).cuda())
    assert np.max(np.abs(logit.cpu().numpy() - z['logit'])) < 1e-4        # north-star fp32 tolerance
    assert np.max(np.abs(prob.cpu().numpy() - z['prob'])) < 1e-5
    # replay through the captured graph gives the same answer
    prob2, logit2 = eng.infer(torch.from_numpy(z['x']).cuda())
    prob3, logit3 = eng.infer(torch.from_numpy(z['x']).cuda())
    assert torch.equal(logit2, logit3) and np.max(np.abs(logit3.cpu().numpy() - z['logit'])) < 1e-4


def test_golden_tta_fp32(cuda, golden_dir):
    z = np.load(golden_dir + '/unet_nfb4_32.npz')
    w = golden_weights(z)
    eng = _engine(4, 'fp32', w)
    mask, act = eng.predict_tta(torch.from_numpy(z['s']).cuda(), window=32)
    assert np.max(np.abs(act.cpu().numpy() - z['tta_act'])) < 1e-5
    flips = (mask.cpu().numpy() != z['tta_mask'])
    assert np.all(np.abs(z['tta_act'][flips] - 0.5) < 1e-5)          # only exact-threshold pixels may differ
    mask1, _ = eng.predict_tta(torch.from_numpy(z['s']).cuda(), window=32, augmentation=False)
    o1, _ = oracle.tta_predict(w, z['s'], oracle.UNetSpec(4), augmentation=False, window=32, dtype=torch.float64)
    assert np.mean(mask1.cpu().numpy() != o1) < 0.002


@pytest.mark.parametrize('loss', ['dice_loss', 'binary_crossentropy', 'dicesq_loss', 'weighted_binary_crossentropy'])
def test_golden_train_step_fp32(cuda, golden_dir, loss):
    z = np.load(golden_dir + '/unet_nfb4_32.npz')
    w = golden_weights(z)
    eng = _engine(4, 'fp32', w, use_graphs=False)
    m = eng.train_step(torch.from_numpy(z['x']).cuda(), torch.from_numpy(z['y']).cuda(), loss=loss, lr=0.002,
                       dropout=False)
    L = float(m[0].item())
    assert abs(L - float(z[loss + ':loss'])) < 1e-4 * max(1.0, abs(L))
    # botb/kernel is compared at the fixture's stored sample of its entries (as_stored), every other tensor in full
    for key in ('enc0a/kernel', 'botb/kernel', 'up2/kernel', 'dec0b/gamma', 'head/kernel', 'head/bias'):
        g_ref = z['%s:grad:%s' % (loss, key)]
        g = as_stored(z, key, eng.G[key].cpu().numpy().astype(np.float64))
        rel = np.linalg.norm(g - g_ref) / (np.linalg.norm(g_ref) + 1e-30)
        assert rel < 2e-3, (key, rel)
    new = eng.get_weights_dict()
    assert np.allclose(new['enc0a/moving_mean'], z[loss + ':new:enc0a/moving_mean'], atol=1e-5)
    assert np.allclose(new['up1/moving_var'], z[loss + ':new:up1/moving_var'], atol=1e-5)
    # Keras-Adam first step moves every weight by lr * sign(g): compare where the gradient is not ~0
    for key in ('botb/kernel', 'head/kernel'):
        g_ref = z['%s:grad:%s' % (loss, key)]
        big = np.abs(g_ref) > 1e-3 * np.abs(g_ref).max()
        assert np.allclose(as_stored(z, key, new[key])[big], z['%s:new:%s' % (loss, key)][big], atol=2e-5), key


def _nfb32_case(seed=7535, shape=(2, 64, 64)):
    spec = oracle.UNetSpec(32)
    w = oracle.init_weights(spec, seed=seed)
    x = np.random.default_rng(865).standard_normal(shape).astype(np.float32)
    return spec, w, x


def test_forward_nfb32_against_oracle_fp32(cuda):
    spec, w, x = _nfb32_case()
    ref = oracle.unet_forward(w, x, spec, dtype=torch.float64)['logit'].numpy()
    eng = _engine(32, 'fp32', w)
    _, logit = eng.infer(torch.from_numpy(x).cuda())
    assert np.abs(logit.cpu().numpy() - ref).max() < 1e-4          # north-star fp32 check-mode tolerance


def test_forward_nfb32_against_oracle_bf16(cuda):
    """bf16 tensor-core mode against two references.
    (1) The oracle with bf16 *storage* emulated at the same points (weights, activations): the first
        layers must agree bit for bit; deeper layers drift apart because a 1-ulp rounding flip fans out
        to 9*Cout outputs per layer (measured: 100 % / 99.97 % / 99.5 % / 95 % / 70 % exact after
        enc0a / enc0b / enc1b / enc2b / botb) - two correct bf16 implementations differ that way.
    (2) The fp64 oracle: the GPU's error must be no larger than the error inherent to bf16 storage,
        i.e. the emulation's own distance from fp64 (both ~1.2e-2 mean on |logit| <= ~7)."""
    spec, w, x = _nfb32_case()
    o64 = oracle.unet_forward(w, x, spec, dtype=torch.float64, return_intermediates=True)
    o16 = oracle.unet_forward(w, x, spec, dtype=torch.float64, emulate_bf16=True, return_intermediates=True)
    eng = _engine(32, 'bf16', w, use_graphs=False)
    _, logit = eng.infer(torch.from_numpy(x).cuda())
    act = eng._sessions[(x.shape[0], x.shape[1], x.shape[2], False)]['act']
    for name, min_exact in (('enc0a', 0.9999), ('enc0b', 0.999), ('enc1a', 0.99)):
        got = act[name].float().cpu().permute(0, 3, 1, 2).double()
        assert float((got == o16['intermediates'][name]).double().mean()) >= min_exact, name
    got = logit.cpu().numpy()
    e_gpu = np.abs(got - o64['logit'].numpy())
    e_emu = np.abs(o16['logit'].numpy() - o64['logit'].numpy())
    print('bf16 logits vs fp64 oracle: GPU max %.4f mean %.5f | bf16-storage emulation max %.4f mean %.5f'
          % (e_gpu.max(), e_gpu.mean(), e_emu.max(), e_emu.mean()))
    assert e_gpu.mean() <= 1.25 * e_emu.mean() + 1e-3
    assert e_gpu.max() <= 1.5 * e_emu.max() + 1e-2
    assert e_gpu.mean() < 2e-2          # the north star's 1e-2 is not reachable with 8-bit mantissas here


def _cudnn_bf16_witness(w, x, spec):
    """An INDEPENDENT 16-bit-storage implementation of the inference graph, checker only: torch / cuDNN conv2d on bf16
    tensors (tensor cores, fp32 accumulate, bf16 output), bias + folded BatchNorm + ReLU in fp32, activations rounded to
    bf16 after every block - the same storage points as the tcgen05 path, none of its code."""
    import torch.nn.functional as F
    dev = torch.device('cuda')
    bf = torch.bfloat16

    def T(a):
        return torch.as_tensor(np.asarray(a, dtype=np.float32), device=dev)

    def block(name, t):
        k = T(w[name + '/kernel'])
        sc = T(w[name + '/gamma']) * torch.rsqrt(T(w[name + '/moving_var']) + 1e-3)
        sh = T(w[name + '/beta']) + (T(w[name + '/bias']) - T(w[name + '/moving_mean'])) * sc
        if name.startswith('up'):
            z = F.conv_transpose2d(t.to(bf), k.permute(3, 2, 0, 1).contiguous().to(bf), stride=2).float()
        else:
            z = F.conv2d(t.to(bf), k.permute(3, 2, 0, 1).contiguous().to(bf), padding=1).float()
        return torch.relu(z * sc[None, :, None, None] + sh[None, :, None, None]).to(bf).float()

    t = T(x)[:, None]
    # first layer: 1 input channel, fp32 arithmetic on the fp32 image like the product's CUDA-core kernel
    k = T(w['enc0a/kernel'])
    sc = T(w['enc0a/gamma']) * torch.rsqrt(T(w['enc0a/moving_var']) + 1e-3)
    sh = T(w['enc0a/beta']) + (T(w['enc0a/bias']) - T(w['enc0a/moving_mean'])) * sc
    t = torch.relu(F.conv2d(t, k.permute(3, 2, 0, 1), padding=1) * sc[None, :, None, None] + sh[None, :, None, None]).to(bf).float()
    skips = []
    t = block('enc0b', t); skips.append(t); t = F.max_pool2d(t, 2)
    for l in (1, 2, 3):
        t = block('enc%db' % l, block('enc%da' % l, t)); skips.append(t); t = F.max_pool2d(t, 2)
    t = block('botb', block('bota', t))
    for l in (3, 2, 1, 0):
        t = torch.cat([block('up%d' % l, t), skips[l]], dim=1)
        t = block('dec%db' % l, block('dec%da' % l, t))
    hk = T(w['head/kernel'])[0, 0]                       # [C, 2]
    hb = T(w['head/bias'])
    z = torch.einsum('nchw,cd->ndhw', t, hk) + hb[None, :, None, None]
    return (z[:, 1] - z[:, 0]).cpu().numpy()


def _keras_random_init(seed=7535):
    """BASELINE config C1's "random-init weights": the product's Keras-style initialiser (truncated he_normal kernels, zero
    biases, gamma 1, beta 0) with randomised moving statistics so that the folded BatchNorm is not the identity"""
    from deepcalcium.engine.graph import GraphSpec, he_normal_weights
    spec = GraphSpec(32)
    w = he_normal_weights(spec, seed=seed)
    rng = np.random.default_rng(seed)
    for blk in spec.blocks:
        if blk.kind != 'head':
            w[blk.name + '/moving_mean'] = (0.1 * rng.standard_normal(blk.cout)).astype(np.float32)
            w[blk.name + '/moving_var'] = rng.uniform(0.5, 1.5, blk.cout).astype(np.float32)
    return w


@pytest.mark.parametrize('case', [('oracle-randomised', (2, 64, 64)), ('oracle-randomised', (1, 512, 512)),
                                  ('keras-init', (1, 512, 512))])
def test_sixteen_bit_logit_error_against_an_independent_cudnn_bf16_witness(cuda, case):
    """North star: logits within 1e-2 absolute in 16-bit mode.  Three implementations against the float64 oracle on the
    same weights and input (512x512 = BASELINE config C1, one summary image):
      * the tcgen05 path with bf16 activations,
      * an independent bf16 witness (torch / cuDNN convolutions on bf16 tensors, same storage points),
      * the tcgen05 path with fp16 activations (kind::f16 runs fp16 operands at the same rate; 3 more mantissa bits).
    bf16 storage cannot meet 1e-2 on a random-init network - two independent bf16 implementations land at the same error,
    6-12x over - while the fp16 mode meets it on the C1 configuration (Keras-style random init) and on the small image
    of the harsher oracle weight set (random gamma / beta / bias); on that set at 512x512 the MAXIMUM over 262 144 pixels
    is 1.4e-2 with 99.98 % of the pixels inside 1e-2 (asserted: >= 99.9 %)."""
    which, shape = case
    allow_tf32 = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        spec, w, _ = _nfb32_case()
        if which == 'keras-init':
            w = _keras_random_init()
        x = np.random.default_rng(865).standard_normal(shape).astype(np.float32)
        with torch.no_grad():
            ref = oracle.unet_forward(w, x, spec, dtype=torch.float64)['logit'].numpy()
        e_wit = np.abs(_cudnn_bf16_witness(w, x, spec) - ref)
        errs = {}
        for precision in ('bf16', 'fp16'):
            eng = _engine(32, precision, w)
            _, logit = eng.infer(torch.from_numpy(x).cuda())
            errs[precision] = np.abs(logit.cpu().numpy() - ref)
    finally:
        torch.backends.cudnn.allow_tf32 = allow_tf32
    frac_in = float(np.mean(errs['fp16'] <= 1e-2))
    print('logit |err| vs fp64 oracle, %s weights at %s (max / mean): tcgen05 bf16 %.4f / %.5f | cuDNN bf16 witness %.4f / %.5f | '
          'tcgen05 fp16 %.4f / %.5f (%.4f %% of pixels within 1e-2) | logit range %.2f'
          % (which, shape, errs['bf16'].max(), errs['bf16'].mean(), e_wit.max(), e_wit.mean(), errs['fp16'].max(),
             errs['fp16'].mean(), 100 * frac_in, np.abs(ref).max()))
    # the two bf16 implementations agree on what bf16 storage costs
    assert errs['bf16'].mean() <= 1.25 * e_wit.mean() + 1e-3
    assert errs['bf16'].max() <= 1.5 * e_wit.max() + 1e-2
    assert e_wit.max() > 2e-2                    # ... and it is not 1e-2
    # the fp16-activation mode
    assert errs['fp16'].mean() <= 2.5e-3 and frac_in >= 0.999 and errs['fp16'].max() <= 2e-2
    if which == 'keras-init' or shape[1] <= 64:
        assert errs['fp16'].max() <= 1e-2, errs['fp16'].max()


def test_forward_512_and_tta_bf16_mask_disagreement(cuda):
    """BASELINE configs C1/C4 shape: one 512x512 summary image, 8x TTA; thresholded mask may differ from
    the fp64 oracle in <= 0.1 % of the pixels (north star)."""
    spec = oracle.UNetSpec(32)
    w = oracle.init_weights(spec, seed=7535)
    s = np.random.default_rng(865).standard_normal((512, 512)).astype(np.float32)
    omask, oact = oracle.tta_predict(w, s, spec, dtype=torch.float32)
    for precision, lim in (('fp32', 1e-4), ('bf16', 1e-3)):
        eng = _engine(32, precision, w)
        mask, act = eng.predict_tta(torch.from_numpy(s).cuda())
        mask = mask.cpu().numpy().copy()          # predict_tta returns static buffers: copy before the next call
        dis = float(np.mean(mask != omask))
        assert dis <= lim, (precision, dis)
        # D4 equivariance property (size independent): rotating the input rotates the TTA output
        mask_r, _ = eng.predict_tta(torch.from_numpy(np.ascontiguousarray(np.rot90(s))).cuda())
        assert np.mean(np.rot90(mask) != mask_r.cpu().numpy()) <= 2 * lim + 1e-5


@pytest.mark.parametrize('fused_bn', [3, 2, 1, 0])
@pytest.mark.parametrize('precision', ['fp32', 'bf16'])
def test_train_step_nfb32_against_oracle(cuda, precision, fused_bn):
    """One train_on_batch (dice, dropout off): loss, every gradient tensor, BN moving statistics.
    fp32 check mode: within 3e-3 relative L2 of the fp64 oracle for every tensor.  (The BN backward of this
    random-init dice network cancels catastrophically - dz - mean(dz) - so even torch-CPU float32 autograd of the
    oracle is 1e-3 away from its own float64 run from dec0a downwards; the check-mode kernels use blocked fp32
    summation and land at 0.7e-3 ... 1.2e-3; measured, see DESIGN.md.)
    bf16 mode: the fp64 gradient of this random-init dice network moves by 20-65 % under 2^-9
    perturbations of the stored activations (measured on CPU with the bf16-storage emulation of the
    oracle), so the criterion is: the GPU's distance from fp64 is no larger than the emulation's own
    distance from fp64 (x1.3 + 0.03), per tensor."""
    spec, w, _ = _nfb32_case()
    rng = np.random.default_rng(865)
    x = rng.standard_normal((4, 32, 32)).astype(np.float32)
    y = (rng.random((4, 32, 32)) < 0.126).astype(np.uint8)
    L, nw, st, g, _ = oracle.train_step(w, x, y, spec=spec, loss='dice_loss')
    from deepcalcium import _native as nat
    eng = _engine(32, precision, w, use_graphs=False)
    # BatchNorm variants: 3 / 2 = batch statistics taken in the conv epilogues (bf16; everywhere / where it pays = the
    # default), 1 = single-launch kernels, 0 = separate passes
    with nat.policy(fused_bn=fused_bn):
        m = eng.train_step(torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda(), loss='dice_loss', dropout=False)
    assert abs(float(m[0].item()) - L) < (1e-4 if precision == 'fp32' else 2e-3)
    if precision == 'bf16':
        _, _, _, g_emu, _ = oracle.train_step(w, x, y, spec=spec, loss='dice_loss', emulate_bf16=True)

    def rel(a, b):
        return np.linalg.norm(a - b) / (np.linalg.norm(b) + 1e-30)

    worst = ('', 0.0)
    for key, g_ref in g.items():
        if key.endswith('/bias') and not key.startswith('head'):
            continue                      # exactly zero by construction (bias feeds a batch-stat BN)
        got = eng.G[key].cpu().numpy().astype(np.float64)
        r = rel(got, g_ref)
        if precision == 'fp32':
            assert r < 3e-3, (key, r)
        else:
            assert r <= 1.3 * rel(g_emu[key], g_ref) + 0.03, (key, r, rel(g_emu[key], g_ref))
        if r > worst[1]:
            worst = (key, r)
    print('%s: worst gradient relative L2 error vs fp64: %s = %.4f' % (precision, worst[0], worst[1]))
    new = eng.get_weights_dict()
    for key in ('enc2b/moving_mean', 'up0/moving_var', 'dec1a/moving_var'):
        assert np.allclose(new[key], nw[key], atol=1e-4 if precision == 'fp32' else 2e-2), key


@pytest.mark.parametrize('precision', ['fp32', 'bf16'])
def test_train_step_at_the_benchmarked_shape_c3(cuda, precision):
    """BASELINE config C3 at its own shape - 32 crops of 128x128, dice loss, dropout off - under the DEFAULT dispatch
    policy and through the CUDA-graph path bench.py times (call 1 eager, call 2 capture + replay): loss, every gradient
    tensor and the BN moving statistics against oracle.train_step (float64).  Same criteria as the small-shape test."""
    from deepcalcium import _native as nat
    nat.reset_policy()
    spec, w, _ = _nfb32_case()
    rng = np.random.default_rng(865)
    x = rng.standard_normal((32, 128, 128)).astype(np.float32)
    y = (rng.random((32, 128, 128)) < 0.126).astype(np.uint8)
    L, nw, st, g, _ = oracle.train_step(w, x, y, spec=spec, loss='dice_loss')
    # yardsticks: bf16 mode - the oracle with bf16 storage emulated; fp32 check mode - the oracle run in float32 on the CPU
    # (torch autograd): at 524 288 pixels per channel the BatchNorm-backward cancellation makes ANY float32 evaluation of
    # the first layers' gradients a few 1e-3 off the float64 one
    if precision == 'bf16':
        g_yard = oracle.train_step(w, x, y, spec=spec, loss='dice_loss', emulate_bf16=True)[3]
    else:
        g_yard = oracle.train_step(w, x, y, spec=spec, loss='dice_loss', dtype=torch.float32)[3]
    xd, yd = torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda()

    def rel(a, b):
        return np.linalg.norm(a - b) / (np.linalg.norm(b) + 1e-30)

    for attempt in ('eager', 'graph'):
        eng = _engine(32, precision, w)
        if attempt == 'graph':         # lr = 0 step first: same weights afterwards, the second call is the captured replay
            eng.train_step(xd, yd, loss='dice_loss', lr=0.0, dropout=False)
            eng.set_weights_dict(w); eng.reset_optimizer()
            eng.train_step(xd, yd, loss='dice_loss', lr=0.0, dropout=False)
            eng.set_weights_dict(w); eng.reset_optimizer()
            m = eng.train_step(xd, yd, loss='dice_loss', lr=0.0, dropout=False)
        else:
            m = eng.train_step(xd, yd, loss='dice_loss', lr=0.002, dropout=False)
        assert abs(float(m[0].item()) - L) < (1e-4 if precision == 'fp32' else 2e-3), attempt
        errs = {}
        for key, g_ref in g.items():
            if key.endswith('/bias') and not key.startswith('head'):
                continue
            errs[key] = (rel(eng.G[key].cpu().numpy().astype(np.float64), g_ref), rel(g_yard[key], g_ref))
        worst = max(errs, key=lambda k: errs[k][0])
        print('C3 %s %s: loss %.6f (oracle %.6f), worst gradient rel. L2 error %s = %.4g (yardstick %.4g); median %.4g (yardstick %.4g)'
              % (precision, attempt, float(m[0].item()), L, worst, errs[worst][0], errs[worst][1],
                 np.median([e[0] for e in errs.values()]), np.median([e[1] for e in errs.values()])))
        for key, (r, ry) in errs.items():
            if precision == 'fp32':
                assert r <= max(3e-3, 2.0 * ry), (attempt, key, r, ry)
            else:
                assert r <= 1.3 * ry + 0.03, (attempt, key, r, ry)
        if attempt == 'eager':
            new = eng.get_weights_dict()
            for key in ('enc0b/moving_mean', 'enc2b/moving_var', 'up0/moving_var', 'dec1a/moving_mean', 'botb/moving_var'):
                assert np.allclose(new[key], nw[key], atol=1e-4 if precision == 'fp32' else 2e-2), key


def test_bf16_training_loss_curve_tracks_the_fp32_check_mode(cuda):
    """25 optimiser steps (dice, Adam 0.002, dropout off, a fixed rotation of 4 batches of 8 x 64 x 64) from the same
    initial weights in the bf16 tensor-core mode and in the fp32 check mode: both losses must fall and the bf16 curve must
    stay close to the fp32 one - the constraint on bf16 training that a single-step gradient comparison cannot give."""
    spec, w, _ = _nfb32_case()
    rng = np.random.default_rng(3)
    xs, ys = [], []
    for i in range(4):
        x = rng.standard_normal((8, 64, 64)).astype(np.float32)
        # a learnable target: blobs where a smoothed version of the input is high
        sm = (x + np.roll(x, 1, 1) + np.roll(x, -1, 1) + np.roll(x, 1, 2) + np.roll(x, -1, 2)) / 5
        xs.append(torch.from_numpy(x).cuda()); ys.append(torch.from_numpy((sm > 0.4).astype(np.uint8)).cuda())
    curves = {}
    for precision in ('fp32', 'bf16'):
        eng = _engine(32, precision, w)
        curves[precision] = [float(eng.train_step(xs[i % 4], ys[i % 4], loss='dice_loss', lr=0.002, dropout=False)[0].item())
                             for i in range(25)]
    f, b = np.array(curves['fp32']), np.array(curves['bf16'])
    print('loss curves fp32 %s\n            bf16 %s' % (np.round(f, 4).tolist(), np.round(b, 4).tolist()))
    assert f[-4:].mean() < f[:4].mean() - 0.05 and b[-4:].mean() < b[:4].mean() - 0.05
    assert np.abs(b[:5] - f[:5]).max() < 5e-3          # the first steps are the same computation up to bf16 rounding
    assert np.abs(b - f).max() < 0.05 and np.abs(b - f).mean() < 0.02


def test_training_graph_replay_decreases_loss_and_matches_eager(cuda):
    spec, w, _ = _nfb32_case()
    rng = np.random.default_rng(1)
    x = rng.standard_normal((4, 32, 32)).astype(np.float32)
    y = (x > 0.5).astype(np.uint8)
    xd, yd = torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda()
    runs = {}
    for graphs in (False, True):
        eng = _engine(32, 'fp32', w, use_graphs=graphs)
        losses = [float(eng.train_step(xd, yd, loss='dice_loss', dropout=False)[0].item()) for _ in range(6)]
        runs[graphs] = losses
        assert losses[-1] < losses[0]
        assert int(eng.step_state[0].item()) == 6
    assert np.allclose(runs[False], runs[True], atol=1e-4)


def test_reference_surface_fit_predict_evaluate(cuda, tmp_path):
    from deepcalcium.models.neurons import UNet2DSummary, unet
    from deepcalcium.models.neurons.unet_2d_summary import Adam
    from deepcalcium.datasets.nf import make_dataset
    rng = np.random.default_rng(0)
    paths = []
    for i in range(2):
        masks = np.zeros((6, 96, 112), np.int8)
        for k in range(6):
            cy, cx = rng.integers(10, 86), rng.integers(10, 100)
            masks[k, cy - 4:cy + 4, cx - 4:cx + 4] = 1
        movie = rng.random((40, 96, 112)).astype(np.float32) * 50 + masks.max(0)[None] * 100 * rng.random((40, 1, 1))
        paths.append(make_dataset(str(tmp_path / ('ds%d.npz' % i)), 'synthetic.%02d' % i, movie=movie, masks=masks))
    np.random.seed(865)
    model = UNet2DSummary(cpdir=str(tmp_path / 'cp'),
                          net_builder_func=lambda shape: unet(shape, nb_filters_base=32, precision='fp32'))
    hist, model_path = model.fit(paths, shape_trn=(32, 32), shape_val=(128, 128), batch_size_trn=4, nb_steps_trn=3,
                                 nb_epochs=2, optimizer=Adam(0.002), loss='dice_loss')
    assert os.path.exists(model_path) and len(hist['loss']) == 2 and 'val_nf_f1_mean' in hist
    with pytest.raises(AssertionError):
        model.predict(paths, model_path, window_shape=(256, 256))        # reference: only 512x512 (:565)
    assert model_path.endswith('.hdf5')                # Keras-layout checkpoints, like the reference's ModelCheckpoint (:423)
    Mp, names = model.predict(paths, model_path, augmentation=True, save=True)
    assert names == ['synthetic.00', 'synthetic.01'] and Mp[0].shape == (96, 112) and Mp[0].dtype == np.uint8
    assert os.path.exists(str(tmp_path / 'cp' / 'synthetic.00_mp.png'))          # outlined figure (:610-619)
    # the checkpoint is a Keras-2.0.6-layout file: same weights back, and a resumed fit keeps the optimizer state
    from deepcalcium.utils.keras_hdf5 import read_keras_weights
    from deepcalcium.models.neurons.unet_2d_summary import load_model_with_new_input_shape
    spec_k, w_k, info = read_keras_weights(model_path)
    assert spec_k.nfb == 32 and len(w_k) == 134 and info['keras_version'] == '2.0.6'
    m2 = load_model_with_new_input_shape(model_path, (32, 32), compile=True, precision='fp32')
    assert int(m2.engine.step_state[0].item()) == 6 and float(m2.engine.adam_v.abs().sum().item()) > 0
    w_back = m2.engine.get_weights_dict()
    assert all(np.array_equal(w_back[k], w_k[k]) for k in w_k)
    scores = model.evaluate(paths, model_path)
    assert set(scores.keys()) == {True, False}


@pytest.mark.parametrize('precision', ['fp32', 'bf16'])
def test_factored_head_gradient_equals_the_materialised_one(cuda, precision):
    """dL/d(dec0b) = gpix[pixel] * wd[channel] kept as its two factors (dcb_head_loss_bwd_rank1 + dcb_bn_train_bwd_rank1, the
    default) against the materialised [N, H, W, 32] gradient: the same products in the same summation order - up to the
    compiler contracting gpix * wd into the multiply-adds that consume it, one fp32 rounding that the cancelling BatchNorm
    sums of this network amplify to ~1e-4 - so: same loss, every gradient tensor within 1e-3 relative L2."""
    spec, w, _ = _nfb32_case()
    rng = np.random.default_rng(11)
    x = torch.from_numpy(rng.standard_normal((4, 64, 64)).astype(np.float32)).cuda()
    y = torch.from_numpy((rng.random((4, 64, 64)) < 0.126).astype(np.uint8)).cuda()
    grads = {}
    for rank1 in (True, False):
        eng = _engine(32, precision, w, use_graphs=False)
        eng.rank1_head_grad = rank1
        m = eng.train_step(x, y, loss='dice_loss', dropout=True)
        grads[rank1] = (float(m[0].item()), {k: v.clone() for k, v in eng.G.items()})
    assert abs(grads[True][0] - grads[False][0]) < 1e-6
    for k in grads[True][1]:
        a, b = grads[True][1][k].double(), grads[False][1][k].double()
        assert float((a - b).norm() / (b.norm() + 1e-30)) < 1e-3, k


def test_pipelined_predict_equals_the_serial_engine_calls(cuda, tmp_path):
    """UNet2DSummary.predict overlaps upload / step / download of consecutive images over two buffer slots
    (unet_2d_summary.py:578-595 is a serial loop): seven different images of two shapes, with and without TTA, must come
    back exactly as engine.predict_tta computes them one at a time, in order."""
    from deepcalcium.models.neurons import UNet2DSummary
    from deepcalcium.models.neurons.unet_2d_summary import UNetModel
    spec, w, _ = _nfb32_case()
    eng = _engine(32, 'fp16', w)
    rng = np.random.default_rng(5)
    imgs = {('img%d' % i): rng.standard_normal((500, 480) if i % 3 else (512, 512)).astype(np.float32) for i in range(7)}
    model = UNetModel.__new__(UNetModel)
    model.window_shape, model.spec, model.engine = (512, 512), spec, eng
    api = UNet2DSummary(cpdir=str(tmp_path / 'cp'), dataset_name_func=lambda p: p, series_summary_func=lambda p: imgs[p])
    paths = list(imgs.keys())
    for aug in (True, False):
        for rep in range(2):                     # second pass: every slot replays its captured graph
            Mp, names = api.predict(paths, model, augmentation=aug)
            assert names == paths
            for p_, mp in zip(paths, Mp):
                m1, _ = eng.predict_tta(torch.from_numpy(imgs[p_]).cuda(), augmentation=aug)
                assert np.array_equal(mp, m1.cpu().numpy()), (aug, rep, p_)


@pytest.mark.parametrize('precision', ['fp32', 'bf16'])
def test_upsampling_mode_forward_and_train_step(cuda, precision):
    """The non-default `upsampling_or_transpose='upsampling'` graph (unet_2d_summary.py:160-161): nearest 2x upsampling
    instead of the transposed conv blocks, concat widths 768 / 384 / 192 / 96.  Forward logits and one training step
    (dropout off) against the oracle, same criteria as the default graph."""
    from deepcalcium.engine.graph import GraphSpec
    from deepcalcium.engine.unet_engine import UNetEngine
    spec = oracle.UNetSpec(32, upsampling_or_transpose='upsampling')
    w = oracle.init_weights(spec, seed=7535)
    assert not any(k.startswith('up') for k in w)
    rng = np.random.default_rng(865)
    x = rng.standard_normal((2, 64, 64)).astype(np.float32)
    y = (rng.random((2, 64, 64)) < 0.126).astype(np.uint8)
    ref = oracle.unet_forward(w, x, spec, dtype=torch.float64)
    eng = UNetEngine(GraphSpec(32, upsampling_or_transpose='upsampling'), precision=precision, use_graphs=False)
    eng.set_weights_dict(w)
    prob, logit = eng.infer(torch.from_numpy(x).cuda())
    err = np.abs(logit.cpu().numpy() - ref['logit'].numpy())
    if precision == 'fp32':
        assert err.max() < 1e-4
    else:
        emu = oracle.unet_forward(w, x, spec, dtype=torch.float64, emulate_bf16=True)
        e_emu = np.abs(emu['logit'].numpy() - ref['logit'].numpy())
        assert err.mean() <= 1.5 * e_emu.mean() + 2e-3 and err.max() <= 2.0 * e_emu.max() + 2e-2
    L, nw, st, g, _ = oracle.train_step(w, x, y, spec=spec, loss='dice_loss')
    m = eng.train_step(torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda(), loss='dice_loss', dropout=False)
    assert abs(float(m[0].item()) - L) < (1e-4 if precision == 'fp32' else 2e-3)
    if precision == 'bf16':
        _, _, _, g_emu, _ = oracle.train_step(w, x, y, spec=spec, loss='dice_loss', emulate_bf16=True)

    def rel(a, b):
        return np.linalg.norm(a - b) / (np.linalg.norm(b) + 1e-30)

    for key, g_ref in g.items():
        if key.endswith('/bias') and not key.startswith('head'):
            continue
        r = rel(eng.G[key].cpu().numpy().astype(np.float64), g_ref)
        if precision == 'fp32':
            assert r < 3e-3, (key, r)
        else:
            assert r <= 1.3 * rel(g_emu[key], g_ref) + 0.03, (key, r, rel(g_emu[key], g_ref))
    # dropout on: the upsampled tensors are masked with keep probability 1 - p and rescaled (mean preserved)
    m2 = eng.train_step(torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda(), loss='dice_loss', dropout=True)
    assert np.isfinite(float(m2[0].item()))
