"""Truth-mask summary on the device (dcb_mask_summary, deepcalcium.datasets.nf.summarize_masks_device) against the
reference's sequential _summarize_mask (oracle/masks.py), bit for bit, and the default plugin of fit / predict against
the host one."""
import numpy as np
import pytest
import torch

import mask_corpus as mc
from oracle.masks import summarize_mask, summarize_mask_array

pytestmark = pytest.mark.gpu


def _dev(m, dtype=None):
    from deepcalcium.datasets.nf import summarize_masks_device
    t = torch.from_numpy(np.ascontiguousarray(m)).cuda()
    out = summarize_masks_device(t if dtype is None else t.to(dtype))
    assert out.dtype == torch.uint8 and out.is_cuda and tuple(out.shape) == m.shape[1:]
    return out.cpu().numpy()


def _check(m):
    got = _dev(m)
    ref = summarize_mask_array(m)
    assert np.array_equal(got.astype(np.float64), ref), (m.shape, int((got != ref).sum()))
    return got


@pytest.mark.parametrize('n', [1, 2, 300, 800, 3000])
def test_random_disks_512(cuda, n):
    m = mc.disks(np.random.default_rng(n), n, 512, 512)
    got = _check(m)
    assert got.sum() > 0


def test_order_sensitive_corpus(cuda):
    for i, m in enumerate(mc.order_corpus()):
        assert np.array_equal(_dev(m).astype(np.float64), summarize_mask_array(m)), i


@pytest.mark.parametrize('shape', [(1, 1), (1, 511), (511, 1), (513, 67), (600, 560)])
def test_shapes(cuda, shape):
    H, W = shape
    rng = np.random.default_rng(H * 1000 + W)
    m = mc.disks(rng, max(2, H * W // 1000), H, W, 1, 9)
    m.flat[rng.integers(0, m.size, m.size // 200 + 1)] = 1      # stray pixels: contested and lone owners
    _check(m)
    _check(m[:1])


def test_no_neurons_and_all_contested(cuda):
    for H, W in ((0, 5), (5, 0), (37, 41)):
        assert np.array_equal(_dev(np.zeros((0, H, W), np.int8)), np.zeros((H, W), np.uint8))
    m = np.ones((3, 45, 70), np.int8)
    assert not _check(m).any()
    m = np.zeros((4, 64, 64), np.int8)                         # every pixel owned by exactly two neurons
    m[0, :32], m[1, :32], m[2, 32:], m[3, 32:] = 1, 1, 1, 1
    assert not _check(m).any()


def test_values_other_than_one_and_dtypes(cuda):
    rng = np.random.default_rng(4)
    base = mc.disks(rng, 60, 128, 96)
    noise = np.array([2, -1, 127, -128], np.int8)[rng.integers(0, 4, base.shape)]
    m8 = np.where(rng.random(base.shape) < 0.05, noise, base).astype(np.int8)
    _check(m8)
    mu8 = m8.view(np.uint8)                                    # -1 -> 255, -128 -> 128
    assert (mu8 == 255).any()
    _check(mu8)
    mb = base.astype(bool)
    _check(mb)
    # bool planes: True is == 1 exactly like the int8 plane it came from
    assert np.array_equal(_dev(base, torch.bool), _dev(base))


def test_owner_ids_above_16_bits(cuda):
    rng = np.random.default_rng(5)
    n, H, W = 70000, 8, 8
    m = np.zeros((n, H, W), np.int8)
    for y in range(H):
        for x in range(W):
            for z in rng.choice(np.arange(60000, n), int(rng.integers(0, 3)), replace=False):   # 0, 1 or 2 owners
                m[z, y, x] = 1
    _check(m)
    solo = np.zeros((n, 4, 4), np.int8)
    solo[65537, 1:3, 1:3] = 1
    solo[1, 0, 0] = 1                                          # touches a neuron whose id differs only above bit 16
    # owner 1's centre (0, 0) comes first and drops (0, 0) and (1, 1); ids cut to 16 bits would look equal and drop nothing
    expect = np.zeros((4, 4), np.uint8)
    expect[1, 2] = expect[2, 1] = expect[2, 2] = 1
    assert np.array_equal(_check(solo), expect)


def test_one_giant_cluster(cuda):
    m = mc.checkerboard(512, 512)
    _, ncand, sizes = mc.decomposed(m)
    assert ncand == 512 * 512 and len(sizes) == 1              # far larger than the shared-memory sort
    _check(m)
    rng = np.random.default_rng(8)
    for k in (2, 5):                                           # random owners: large clusters whose order matters
        m = (rng.random((k, 300, 300)) < 1.0 / k).astype(np.int8)
        _, _, sizes = mc.decomposed(m)
        assert sizes.max() > 2048, sizes.max()
        _check(m)


def test_diagonal_chain(cuda):
    m = mc.diagonal_chain(250, 512, 512, size=5, step=2)
    _, ncand, sizes = mc.decomposed(m)
    assert len(sizes) == 1 and ncand > 900, (ncand, sizes)
    _check(m)


def test_repeated_calls_are_identical(cuda):
    m = mc.disks(np.random.default_rng(6), 800, 512, 512)
    t = torch.from_numpy(m).cuda()
    from deepcalcium.datasets.nf import summarize_masks_device
    first = summarize_masks_device(t)
    for _ in range(5):
        assert torch.equal(summarize_masks_device(t), first)


def test_bad_inputs_are_rejected(cuda):
    from deepcalcium.datasets.nf import summarize_masks_device
    m = torch.zeros(3, 8, 8, dtype=torch.int8, device='cuda')
    for bad in (m.float(), m.to(torch.int16), m.to(torch.int32)):
        with pytest.raises(TypeError):
            summarize_masks_device(bad)
    with pytest.raises(TypeError):
        summarize_masks_device(m.cpu())
    for bad in (m[0], m[None], m.reshape(-1)):
        with pytest.raises(ValueError):
            summarize_masks_device(bad)


# ------------------------------------------------------------------------------------------------- the default plugin
def _datasets(tmp_path, specs):
    from deepcalcium.datasets.nf import make_dataset
    paths = []
    for i, (n, H, W, ext) in enumerate(specs):
        rng = np.random.default_rng(100 + i)
        masks = mc.disks(rng, n, H, W, 3, 7)
        mean = (rng.random((H, W)) * 50 + masks.max(0) * 100).astype(np.float32)
        paths.append(make_dataset(str(tmp_path / ('ds%d.%s' % (i, ext))), 'synthetic.%02d' % i, mean=mean, mx=mean,
                                  masks=masks))
    return paths


def test_summarize_mask_plugin_equals_the_host_function(cuda, tmp_path):
    from deepcalcium.models.neurons.unet_2d_summary import _summarize_mask
    for p in _datasets(tmp_path, [(300, 512, 512, 'hdf5'), (300, 512, 512, 'npz'), (40, 120, 77, 'hdf5')]):
        got, ref = _summarize_mask(p), summarize_mask(p)
        assert got.dtype == ref.dtype == np.float64 and got.shape == ref.shape and np.array_equal(got, ref), p


def test_fit_and_predict_with_the_default_plugin_equal_the_host_plugin(cuda, tmp_path):
    from deepcalcium.models.neurons import UNet2DSummary, unet
    from deepcalcium.models.neurons.unet_2d_summary import Adam, _summarize_mask
    paths = _datasets(tmp_path, [(120, 256, 256, 'hdf5'), (90, 200, 240, 'npz')])
    runs = {}
    for name, func in (('device', _summarize_mask), ('host', summarize_mask)):
        seen = []

        def plugin(p, func=func, seen=seen):
            m = func(p)
            seen.append(m)
            return m
        np.random.seed(865)
        api = UNet2DSummary(cpdir=str(tmp_path / ('cp_' + name)), mask_summary_func=plugin,
                            net_builder_func=lambda shape: unet(shape, nb_filters_base=8, precision='bf16', seed=3))
        hist, model_path = api.fit(paths, shape_trn=(64, 64), shape_val=(256, 256), batch_size_trn=4, nb_steps_trn=3,
                                   nb_epochs=2, optimizer=Adam(0.002), loss='dice_loss')
        api.predict(paths, model_path, print_scores=True, save=True)
        runs[name] = (hist, dict(api.last_scores), seen)
    (hd, sd, md), (hh, sh, mh) = runs['device'], runs['host']
    # fit summarises each dataset once; predict with print_scores and save once more (the figure reuses the summary)
    assert len(md) == len(mh) == 2 * len(paths)
    assert all(a.dtype == b.dtype == np.float64 and np.array_equal(a, b) for a, b in zip(md, mh))
    assert hd.keys() == hh.keys() and all(np.array_equal(hd[k], hh[k], equal_nan=True) for k in hh), (hd, hh)
    assert sd.keys() == sh.keys() and all(np.array_equal(sd[k], sh[k], equal_nan=True) for k in sh), (sd, sh)
