"""nb_filters_base other than 32 in the 16-bit tensor-core modes: the engine runs them on zero-padded channels
(graph.padded_width).  Forward and training step against the oracle under the nfb-32 criteria of test_gpu_unet.py, the
zero invariant of the padded entries over many replayed steps, checkpoints across precisions, the reference surface at
the default precision, and the tiled path."""
import gc
import os

import numpy as np
import pytest
import torch

import oracle
from deepcalcium.engine.graph import GraphSpec, flat_layout, pack_flat, plan_tiles, unpack
from deepcalcium.utils.neurons import INVERTIBLE_2D_AUGMENTATIONS

pytestmark = pytest.mark.gpu

MODES = ('transpose', 'upsampling')


def _engine(nfb, precision, w, mode='transpose', **kw):
    from deepcalcium.engine.unet_engine import UNetEngine
    eng = UNetEngine(GraphSpec(nfb, upsampling_or_transpose=mode), precision=precision, **kw)
    eng.set_weights_dict(w)
    return eng


def _case(nfb, mode='transpose', seed=7535):
    spec = oracle.UNetSpec(nfb, upsampling_or_transpose=mode)
    return spec, oracle.init_weights(spec, seed=seed)


def _rel(a, b):
    return np.linalg.norm(a - b) / (np.linalg.norm(b) + 1e-30)


def _real_channels(eng, name):
    """channels of session tensor ``name`` that hold real values (the rest are padding)"""
    spec = eng.spec
    if name in spec.by_name:
        return spec.by_name[name].cout
    if name.startswith('pool'):
        return spec.by_name['enc%sb' % name[4:]].cout
    return spec.cat_split['dec%sa' % name[2:]]              # nearest-upsampled tensor of the 'upsampling' graph


@pytest.mark.parametrize('mode', MODES)
@pytest.mark.parametrize('nfb', [8, 16, 24, 48, 64])
def test_forward_against_oracle(cuda, nfb, mode):
    """bf16: no further from the fp64 oracle than the oracle's own bf16-storage emulation (the relative criteria of
    test_forward_nfb32_against_oracle_bf16).  The absolute bounds of the nfb-32 tests (bf16 mean < 2e-2, fp16 max <= 1e-2)
    do not carry over: on these random-init weights the bf16-storage emulation itself - no GPU code involved - is up to
    0.04 (mean) / 0.25 (max) from fp64 at some widths.  fp16 keeps 3 more mantissa bits, so its error is held to the
    emulation's scaled by 2^-3 (with room for the rounding of a different summation order): mean <= 0.2x, max <= 0.25x.
    The padded channels of every activation are exactly 0."""
    spec, w = _case(nfb, mode)
    x = np.random.default_rng(865).standard_normal((2, 64, 64)).astype(np.float32)
    o64 = oracle.unet_forward(w, x, spec, dtype=torch.float64)['logit'].numpy()
    e_emu = np.abs(oracle.unet_forward(w, x, spec, dtype=torch.float64, emulate_bf16=True)['logit'].numpy() - o64)
    errs = {}
    for precision in ('bf16', 'fp16'):
        eng = _engine(nfb, precision, w, mode, use_graphs=False)
        _, logit = eng.infer(torch.from_numpy(x).cuda())
        errs[precision] = np.abs(logit.cpu().numpy() - o64)
        for name, a in eng._sessions[(2, 64, 64, False)]['act'].items():
            assert not bool(a[..., _real_channels(eng, name):].any()), (precision, name)
    print('nfb %d %s: logit |err| vs fp64 (max / mean): bf16 %.4f / %.5f, bf16 emulation %.4f / %.5f, fp16 %.4f / %.5f'
          % (nfb, mode, errs['bf16'].max(), errs['bf16'].mean(), e_emu.max(), e_emu.mean(), errs['fp16'].max(),
             errs['fp16'].mean()))
    assert errs['bf16'].mean() <= 1.25 * e_emu.mean() + 1e-3
    assert errs['bf16'].max() <= 1.5 * e_emu.max() + 1e-2
    assert errs['fp16'].mean() <= 0.2 * e_emu.mean() and errs['fp16'].max() <= 0.25 * e_emu.max()


@pytest.mark.parametrize('nfb', [8, 16, 24, 48, 64])
def test_tta_512_mask_disagreement_with_the_fp32_check_mode(cuda, nfb):
    """fp16, the inference precision: the 0.1 % bound of test_forward_512_and_tta_bf16_mask_disagreement.  bf16 storage
    flips up to 0.15 % of these masks at nfb 16 / 24, where its logit error is that of the bf16-storage emulation (see
    test_forward_against_oracle): 0.2 %."""
    spec, w = _case(nfb)
    s = torch.from_numpy(np.random.default_rng(865).standard_normal((512, 512)).astype(np.float32)).cuda()
    ref = _engine(nfb, 'fp32', w).predict_tta(s)[0].cpu().numpy().copy()
    for precision in ('bf16', 'fp16'):
        mask = _engine(nfb, precision, w).predict_tta(s)[0].cpu().numpy()
        dis = float(np.mean(mask != ref))
        print('nfb %d %s: 8x TTA mask disagreement with fp32 %.5f' % (nfb, precision, dis))
        assert dis <= (1e-3 if precision == 'fp16' else 2e-3), (precision, dis)


@pytest.mark.parametrize('nfb', [16, 64])
def test_train_step_against_oracle_bf16(cuda, nfb):
    """one dice step, dropout off, against the fp64 oracle with the oracle's bf16-storage emulation as the yardstick
    (test_train_step_nfb32_against_oracle): loss within 2e-3, moving statistics within 2e-2, every gradient tensor no
    further from fp64 than the emulation is (x1.3 + 0.03 at the median over tensors, x1.5 + 0.03 for each tensor: the
    bf16 gradient of this random-init dice network moves by tens of percent under one bf16 rounding of the stored
    activations, so single tensors of two bf16 evaluations scatter around each other)"""
    spec, w = _case(nfb)
    rng = np.random.default_rng(865)
    x = rng.standard_normal((4, 32, 32)).astype(np.float32)
    y = (rng.random((4, 32, 32)) < 0.126).astype(np.uint8)
    L, nw, _, g, _ = oracle.train_step(w, x, y, spec=spec, loss='dice_loss')
    g_emu = oracle.train_step(w, x, y, spec=spec, loss='dice_loss', emulate_bf16=True)[3]
    eng = _engine(nfb, 'bf16', w, use_graphs=False)
    m = eng.train_step(torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda(), loss='dice_loss', dropout=False)
    assert abs(float(m[0].item()) - L) < 2e-3
    grads = unpack(eng.spec, eng.dspec, {k: v.cpu().numpy() for k, v in eng.G.items()})
    errs = {key: (_rel(grads[key].astype(np.float64), g_ref), _rel(g_emu[key], g_ref)) for key, g_ref in g.items()
            if not (key.endswith('/bias') and not key.startswith('head'))}
    for key, (r, r_emu) in errs.items():
        print('nfb %d %-18s gradient rel. L2 error vs fp64: GPU %.4f, bf16 emulation %.4f' % (nfb, key, r, r_emu))
    assert all(r <= 1.5 * r_emu + 0.03 for r, r_emu in errs.values())
    assert np.median([e[0] for e in errs.values()]) <= 1.3 * np.median([e[1] for e in errs.values()]) + 0.03
    new = eng.get_weights_dict()
    for key in ('enc2b/moving_mean', 'up0/moving_var', 'dec1a/moving_var'):
        assert np.allclose(new[key], nw[key], atol=2e-2), key


@pytest.mark.parametrize('mode', MODES)
@pytest.mark.parametrize('nfb', [16, 24])
def test_padded_entries_stay_zero_over_replayed_steps(cuda, nfb, mode):
    """20 graph-replayed bf16 steps with dropout on: every padded entry of the parameters, gradients, Adam moments and
    moving means is exactly 0, and so is every padded channel of the session's activations and (BatchNorm-input)
    gradients"""
    spec, w = _case(nfb, mode)
    eng = _engine(nfb, 'bf16', w, mode)
    rng = np.random.default_rng(2)
    x = torch.from_numpy(rng.standard_normal((8, 64, 64)).astype(np.float32)).cuda()
    y = torch.from_numpy((rng.random((8, 64, 64)) < 0.2).astype(np.uint8)).cuda()
    losses = [float(eng.train_step(x, y, loss='dice_loss', dropout=True)[0].item()) for _ in range(20)]
    assert all(np.isfinite(losses)) and losses[-1] < losses[0]
    torch.cuda.synchronize()
    slots, n_t, _ = flat_layout(eng.spec)
    real = pack_flat(eng.spec, eng.dspec, np.ones(n_t, np.float32)) == 1
    for name in ('params', 'grads', 'adam_m', 'adam_v'):
        t = getattr(eng, name).cpu().numpy()
        assert not t[~real].any(), name
        assert t[real].any(), name
    for key, (tr, _, _) in slots.items():
        if key.endswith('/moving_mean'):
            assert not eng.P[key][eng.spec.by_name[key.split('/')[0]].cout:].any(), key
    s = eng._sessions[(8, 64, 64, True)]
    for part in ('act', 'raw'):
        for name, a in s[part].items():
            if name == 'x':
                continue
            assert not bool(a[..., _real_channels(eng, name):].any()), (part, name)


def _tiny_batch(seed):
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((4, 64, 64)).astype(np.float32)
    return x, (rng.random((4, 64, 64)) < 0.2).astype(np.uint8)


def test_checkpoints_move_between_precisions(cuda, tmp_path):
    from deepcalcium.models.neurons import unet
    from deepcalcium.models.neurons.unet_2d_summary import Adam, load_model_with_new_input_shape
    model = unet((64, 64), nb_filters_base=16, seed=4)
    assert model.engine.precision == 'bf16'
    model.compile(optimizer=Adam(0.002), loss='dice_loss')
    for i in range(3):
        model.train_on_batch(*_tiny_batch(i))
    w0 = model.get_weights()
    st0 = model.engine.get_optimizer_state()
    assert len(w0) == 134 and w0[0].shape == (3, 3, 1, 16)
    assert st0['adam_m'].shape == (flat_layout(GraphSpec(16))[1],) and st0['step_state'][0] == 3
    for ext in ('hdf5', 'npz'):
        model.save(str(tmp_path / ('m.' + ext)))
    xb, yb = _tiny_batch(9)
    ref_metrics = model.train_on_batch(xb, yb)
    ref_w, ref_st = model.get_weights(), model.engine.get_optimizer_state()
    for ext in ('hdf5', 'npz'):
        path = str(tmp_path / ('m.' + ext))
        for precision in ('fp32', 'fp16', 'bf16'):
            m2 = load_model_with_new_input_shape(path, (64, 64), compile=True, precision=precision)
            assert m2.engine.precision == precision
            assert all(np.array_equal(a, b) for a, b in zip(m2.get_weights(), w0)), (ext, precision)
            st = m2.engine.get_optimizer_state()
            assert all(np.array_equal(st[k], st0[k]) for k in st0), (ext, precision)
            assert m2.engine.iteration == 3
        # the next step after the bf16 reload is the next step taken in memory
        assert m2.loss == 'dice_loss'
        assert m2.train_on_batch(xb, yb) == ref_metrics, ext
        assert all(np.array_equal(u, v) for u, v in zip(m2.get_weights(), ref_w)), ext
        st = m2.engine.get_optimizer_state()
        assert all(np.array_equal(st[k], ref_st[k]) for k in ref_st), ext


def test_reference_surface_at_nfb16_default_precision(cuda, tmp_path):
    from deepcalcium.models.neurons import UNet2DSummary, unet
    from deepcalcium.models.neurons.unet_2d_summary import Adam
    from deepcalcium.datasets.nf import make_dataset
    from deepcalcium.utils.keras_hdf5 import read_keras_weights
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
    model = UNet2DSummary(cpdir=str(tmp_path / 'cp'), net_builder_func=lambda shape: unet(shape, nb_filters_base=16))
    hist, model_path = model.fit(paths, shape_trn=(32, 32), shape_val=(128, 128), batch_size_trn=4, nb_steps_trn=3,
                                 nb_epochs=2, optimizer=Adam(0.002), loss='dice_loss')
    assert os.path.exists(model_path) and len(hist['loss']) == 2 and all(np.isfinite(hist['loss']))
    spec_k, w_k, _ = read_keras_weights(model_path)
    assert spec_k.nfb == 16 and len(w_k) == 134 and w_k['dec0b/kernel'].shape == (3, 3, 16, 16)
    Mp, names = model.predict(paths, model_path, augmentation=True)
    assert names == ['synthetic.00', 'synthetic.01'] and Mp[0].shape == (96, 112) and Mp[0].dtype == np.uint8
    scores = model.evaluate(paths, model_path)
    assert set(scores.keys()) == {True, False}


def test_tiled_nfb16_against_the_whole_canvas(cuda):
    """the criteria of test_tiled_fp16_against_the_whole_canvas at 1300 x 900"""
    spec, w = _case(16)
    eng = _engine(16, 'fp16', w)
    s = np.random.default_rng(5).standard_normal((1300, 900)).astype(np.float32)
    plan = plan_tiles(s.shape, eng.halo, 512)
    c = np.pad(s, ((0, plan.canvas[0] - s.shape[0]), (0, plan.canvas[1] - s.shape[1])), mode='reflect')[None]
    ref = np.zeros(s.shape)
    for _, aug, inv in INVERTIBLE_2D_AUGMENTATIONS:
        prob, _ = eng.infer(torch.from_numpy(np.ascontiguousarray(aug(c))).cuda())
        ref += inv(prob.cpu().numpy())[0, :s.shape[0], :s.shape[1]] / np.float32(len(INVERTIBLE_2D_AUGMENTATIONS))
    mask, act = eng.predict_tiled(torch.from_numpy(s).cuda(), tile=512)
    err = float(np.max(np.abs(act.cpu().numpy() - ref)))
    dis = float(np.mean(mask.cpu().numpy() != (ref > 0.5)))
    print('tiled fp16 nfb 16 (%d tiles): max |act diff| %.3g, mask disagreement %.5f' % (plan.n_tiles, err, dis))
    assert err < 1e-2 and dis <= 1e-3


def test_tiled_2048_at_nfb64_peaks_no_higher_than_nfb32(cuda):
    s = torch.from_numpy(np.random.default_rng(6).standard_normal((2048, 2048)).astype(np.float32)).cuda()
    peak = {}
    for nfb in (32, 64):
        gc.collect()
        torch.cuda.empty_cache()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        eng = _engine(nfb, 'fp16', _case(nfb)[1])
        mask, act = eng.predict_tiled(s)
        torch.cuda.synchronize()
        peak[nfb] = torch.cuda.max_memory_allocated() - base
        assert bool(torch.isfinite(act).all())
        print('nfb %d: 2048^2 tiled prediction, tile %d, %d batch pixels per group: peak %.2f GiB'
              % (nfb, eng.max_tile, eng.tile_batch_pixels, peak[nfb] / 2 ** 30))
        del eng, mask, act
    assert peak[64] <= peak[32]
