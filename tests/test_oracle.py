"""Oracle self-tests (CPU): algebraic identities of the restated reference arithmetic and the
committed known-answer fixtures.  PARITY UNPINNED - the reference has no golden vectors."""
import numpy as np
import pytest
import torch

import oracle
from oracle import losses as ol
from oracle.make_golden import as_stored, golden_weights
from oracle.unet import _convT2x2, keras_adam_update


def test_tta_table_is_eight_distinct_invertible_dihedral_maps():
    x = np.arange(2 * 5 * 5, dtype=np.float32).reshape(2, 5, 5)
    seen = []
    for name, aug, inv in oracle.INVERTIBLE_2D_AUGMENTATIONS:
        a = aug(x)
        assert np.array_equal(inv(a), x), name
        seen.append(a.tobytes())
    assert len(set(seen)) == 8
    # rot90vflip == transpose, rot90hflip == anti-transpose (SURVEY section 4)
    t = dict((n, a) for n, a, _ in oracle.INVERTIBLE_2D_AUGMENTATIONS)
    assert np.array_equal(t['rot90vflip'](x), x.transpose(0, 2, 1))
    assert np.array_equal(t['rot90hflip'](x), x[:, ::-1, ::-1].transpose(0, 2, 1))


def test_softmax_last_channel_is_sigmoid_of_logit_difference():
    z = torch.randn(3, 2, 7, 7, dtype=torch.float64)
    p = torch.softmax(z, dim=1)[:, -1]
    assert torch.allclose(p, torch.sigmoid(z[:, 1] - z[:, 0]), atol=1e-14)


def test_conv_transpose_is_gemm_plus_pixel_shuffle():
    rng = np.random.default_rng(0)
    cin, cout = 6, 5
    x = torch.tensor(rng.standard_normal((2, cin, 3, 4)))
    k = torch.tensor(rng.standard_normal((2, 2, cout, cin)))      # Keras layout (kh,kw,Cout,Cin)
    b = torch.tensor(rng.standard_normal(cout))
    ref = _convT2x2(x, k, b)
    out = torch.zeros(2, cout, 6, 8, dtype=torch.float64)
    for a in range(2):
        for c in range(2):
            out[:, :, a::2, c::2] = torch.einsum('nihw,oi->nohw', x, k[a, c]) + b[None, :, None, None]
    assert torch.allclose(ref, out, atol=1e-12)


def test_keras_adam_first_step_moves_by_lr_times_sign():
    p = np.array([1.0, -2.0, 3.0]); g = np.array([0.5, -1e-3, 2.0])
    p1, m1, v1 = keras_adam_update(p, g, np.zeros(3), np.zeros(3), 0, lr=0.002)
    assert np.allclose(p - p1, 0.002 * np.sign(g), rtol=1e-3)
    # epsilon sits outside the bias correction: a zero gradient leaves the parameter alone
    p2, _, _ = keras_adam_update(p, np.zeros(3), np.zeros(3), np.zeros(3), 0)
    assert np.array_equal(p2, p)


def test_bn_inference_uses_eps_1e_3_and_moving_stats():
    spec = oracle.UNetSpec(nb_filters_base=4)
    w = oracle.init_weights(spec, seed=1)
    x = np.random.default_rng(2).standard_normal((1, 16, 16)).astype(np.float32)
    o = oracle.unet_forward(w, x, spec, return_intermediates=True)
    raw, y = o['intermediates']['enc0a/raw'], o['intermediates']['enc0a']
    g, b = (torch.tensor(w['enc0a/' + k], dtype=torch.float64) for k in ('gamma', 'beta'))
    mm, mv = (torch.tensor(w['enc0a/' + k], dtype=torch.float64) for k in ('moving_mean', 'moving_var'))
    exp = torch.relu((raw - mm[None, :, None, None]) / torch.sqrt(mv + 1e-3)[None, :, None, None]
                     * g[None, :, None, None] + b[None, :, None, None])
    assert torch.allclose(exp, y, atol=1e-12)


def test_dice_loss_gradient_formula():
    # the closed form the CUDA head kernel uses (SURVEY 8a row a7)
    rng = np.random.default_rng(5)
    yt = torch.tensor((rng.random(50) < 0.3).astype(np.float64))
    p = torch.tensor(rng.random(50), requires_grad=True)
    ol.dice_loss(yt, p).backward()
    I, D = (yt * p).sum().item(), (yt.sum() + p.sum() + 1e-7).item()
    assert np.allclose(p.grad.numpy(), -2 * (yt.numpy() * D - I) / D ** 2, atol=1e-12)


def test_projection_oracle_and_reference_fp16_artifact():
    rng = np.random.default_rng(7)
    movie = rng.poisson(100, size=(300, 6, 6)).astype(np.int16)
    mean, mx = oracle.project_mean_max(movie)
    assert np.array_equal(mx, movie.max(0).astype(np.float32))
    assert np.allclose(mean, movie.astype(np.float64).mean(0), rtol=1e-7)
    m16, mx16 = oracle.project_streaming_fp16(movie)
    assert np.array_equal(mx16, movie.max(0))
    # the reference's fp16 running mean drifts from the true mean; both stay in the same ballpark
    assert np.all(np.abs(m16.astype(np.float64) - mean) / mean < 0.2)


def test_golden_projection(golden_dir):
    z = np.load(golden_dir + '/projection_small.npz')
    mean, mx = oracle.project_mean_max(z['movie'])
    assert np.array_equal(mean, z['mean']) and np.array_equal(mx, z['max'])
    assert np.allclose(oracle.summarize_series(mean.astype(np.float16)), z['summary'], atol=1e-6)


def test_golden_unet_forward_tta_train(golden_dir):
    z = np.load(golden_dir + '/unet_nfb4_32.npz')
    spec = oracle.UNetSpec(nb_filters_base=4)
    w = golden_weights(z)
    o = oracle.unet_forward(w, z['x'], spec)
    assert np.allclose(o['logit'].numpy(), z['logit'], atol=1e-10)
    mask, act = oracle.tta_predict(w, z['s'], spec, window=32, dtype=torch.float64)
    assert np.array_equal(mask, z['tta_mask']) and np.allclose(act, z['tta_act'], atol=1e-9)
    L, nw, st, g, _ = oracle.train_step(w, z['x'], z['y'], spec=spec, loss='dice_loss')
    assert abs(L - float(z['dice_loss:loss'])) < 1e-10
    assert np.allclose(as_stored(z, 'botb/kernel', g['botb/kernel']), z['dice_loss:grad:botb/kernel'], atol=1e-12)
    assert np.allclose(nw['head/kernel'], z['dice_loss:new:head/kernel'], atol=1e-7)


def test_weight_list_order_is_keras_get_weights_order():
    spec = oracle.UNetSpec()
    w = oracle.init_weights(spec)
    lst = oracle.weights_to_keras_list(w, spec)
    assert len(lst) == 134 and sum(a.size for a in lst) == 7773250
    assert lst[0].shape == (3, 3, 1, 32) and lst[1].shape == (32,) and lst[-2].shape == (1, 1, 32, 2)
    back = oracle.keras_list_to_weights(lst, spec)
    assert all(np.array_equal(back[k], w[k]) for k in w)


# ------------------------------------------------------------------ N3: neurofinder-style scoring (datasets/nf.py:153-229)
def test_nf_mask_metrics_known_answers():
    """Region matching of `neurofinder.centers` / `shapes` (restated, third-party package absent) on hand-computed cases."""
    import sys, os
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'deep-calcium_b200'))
    from deepcalcium.datasets.nf import nf_mask_metrics, _label_regions
    m = np.zeros((40, 40), np.uint8)
    m[5:10, 5:10] = 1; m[20:26, 20:26] = 1; m[30:33, 3:6] = 1
    assert nf_mask_metrics(m, m) == (1.0, 1.0, 1.0, 1.0, 1.0)
    assert nf_mask_metrics(m, np.zeros_like(m)) == (0., 0., 0., 0., 0.)
    mp = np.zeros_like(m)
    mp[6:11, 5:10] = 1          # region 1 shifted one row: overlap 20 / 25
    mp[20:26, 22:28] = 1        # region 2 shifted two columns: overlap 24 / 36
    p, r, i, e, f1 = nf_mask_metrics(m, mp)
    assert p == 1.0 and abs(r - 2. / 3) < 1e-12 and abs(i - (0.8 + 2. / 3) / 2) < 1e-12 and abs(e - i) < 1e-12
    assert abs(f1 - 0.8) < 1e-12
    far = np.zeros_like(m); far[5:10, 15:20] = 1     # centre 10 px away: beyond the 5 px threshold -> no match
    p, r, i, e, f1 = nf_mask_metrics(m, far)
    assert p == 0.0 and r == 0.0 and (i, e) == (0.0, 0.0) and np.isnan(f1)
    # 8-connectivity (skimage.measure.label default in 2-D): diagonal neighbours are one region
    d = np.zeros((6, 6), np.uint8); d[1, 1] = d[2, 2] = d[3, 3] = 1; d[0, 5] = 1
    regs = _label_regions(d)
    assert [len(x) for x in regs] == [1, 3] and regs[0].tolist() == [[0, 5]]


def test_nf_submit_is_bug_compatible(tmp_path):
    import sys, os, json
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'deep-calcium_b200'))
    from deepcalcium.datasets.nf import nf_submit
    m = np.zeros((10, 10), np.uint8); m[1:3, 1:3] = 1; m[6:8, 6:9] = 1
    path = str(tmp_path / 'sub.json')
    nf_submit([m, np.zeros_like(m)], ['neurofinder.00.00', 'x'], path)
    sub = json.load(open(path))
    assert sub[0]['dataset'] == '00.00' and len(sub[0]['regions']) == 1      # range(1, max) drops the last region
    assert sub[0]['regions'][0]['coordinates'] == [[1, 1], [1, 2], [2, 1], [2, 2]]
    assert sub[1]['regions'] == [{'coordinates': [[[0, 0]]]}]
