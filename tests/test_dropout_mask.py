"""The host statement of the dropout keep mask (tests/dropout_mask.py), which the GPU tests hold every mask-drawing kernel
to: Philox4x32-10 against the Random123 known-answer vectors, the threshold and scale, the element order, the statistics
of the mask, and the engine's layer-id / seed / padded-width rules.  No GPU needed."""
import numpy as np
import pytest
import torch

import dropout_mask as dm

SEED = 0x1234567887654321          # both 32-bit halves nonzero
SEED_DEV = 0x0F1E2D3C4B5A6978


@pytest.mark.parametrize('ctr, key, want', [
    ((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
    ((0xffffffff,) * 4, (0xffffffff,) * 2, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
    ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0), (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1)),
])
def test_philox_known_answer_vectors(ctr, key, want):
    assert tuple(int(w) for w in dm.philox4x32_10(*ctr, *key)) == want
    # the vectorised form gives every lane the scalar answer
    got = dm.philox4x32_10(*(np.full(5, c, np.uint64) for c in ctr), *key)
    assert all(np.all(g == w) for g, w in zip(got, want))


def test_element_order_within_a_philox_call():
    """element e = half-word e % 8 of the call for counter e / 8: x low, x high, y low, ... w high"""
    n = 8 * 5 + 3
    u = dm.uniforms16(SEED, 21, n)
    assert u.shape == (n,) and u.dtype == np.uint32
    for g in range(6):
        x, y, z, w = (int(v) for v in dm.philox4x32_10(g, 0, 21, 0, SEED & 0xffffffff, SEED >> 32))
        want = [x & 0xffff, x >> 16, y & 0xffff, y >> 16, z & 0xffff, z >> 16, w & 0xffff, w >> 16]
        assert u[8 * g:8 * g + 8].tolist() == want[:len(u[8 * g:8 * g + 8])]


@pytest.mark.parametrize('p, thr, value', [(0.25, 16384, np.float32(4.0 / 3.0)), (0.5, 32768, np.float32(2.0))])
def test_threshold_and_keep_value(p, thr, value):
    assert dm.threshold(p) == thr
    assert dm.keep_value(p) == value and dm.keep_value(p).dtype == np.float32
    n = 1 << 18
    u = dm.uniforms16(SEED, 17, n)
    k = dm.keep_scale(SEED, 17, n, p)
    assert k.dtype == np.float32 and set(np.unique(k).tolist()) == {0.0, float(value)}
    assert np.array_equal(k > 0, u >= thr)
    # the threshold itself is kept, one below it is dropped (each occurs ~4 times in 2^18 draws)
    assert np.any(u == thr) and np.all(k[u == thr] > 0)
    assert np.any(u == thr - 1) and np.all(k[u == thr - 1] == 0)


def _sigma5(q, n):
    return 5 * np.sqrt(q * (1 - q) / n)


@pytest.mark.parametrize('p', [0.25, 0.5])
def test_keep_fraction_and_independence(p):
    n = 1 << 20
    base = dm.keep_scale(SEED, 17, n, p) > 0
    assert abs(base.mean() - (1 - p)) < _sigma5(1 - p, n)
    # two independent masks agree with probability p^2 + (1-p)^2
    q = p * p + (1 - p) * (1 - p)
    others = {'layer': dm.keep_scale(SEED, 18, n, p), 'seed': dm.keep_scale(SEED + 0x100000001, 17, n, p),
              'device seed': dm.keep_scale(SEED ^ SEED_DEV, 17, n, p)}
    for what, k in others.items():
        agree = float(np.mean((k > 0) == base))
        assert abs(agree - q) < _sigma5(q, n), (what, agree, q)
    # and neither half of the mask is a copy of the other (the two halves of a 32-bit word are not correlated)
    u = dm.uniforms16(SEED, 17, n).reshape(-1, 2)
    lo, hi = u[:, 0] >= dm.threshold(p), u[:, 1] >= dm.threshold(p)
    assert abs(float(np.mean(lo == hi)) - q) < _sigma5(q, n // 2)


def _cpu_engine(nfb, precision, mode='transpose', rank=None, step_seed=0):
    """a UNetEngine with only the graph and the step state: enough for the mask rules, no device"""
    from deepcalcium.engine.graph import GraphSpec
    from deepcalcium.engine.unet_engine import UNetEngine
    eng = UNetEngine.__new__(UNetEngine)
    eng.spec = GraphSpec(nfb, upsampling_or_transpose=mode)
    eng.dspec = eng.spec.device_spec(precision)
    eng._inputs = eng._wire()
    eng.comm = None if rank is None else type('Comm', (), {'rank': rank, 'world': rank + 1})()
    eng.step_state = torch.tensor([1, step_seed - (1 << 64) if step_seed >= 1 << 63 else step_seed], dtype=torch.int64)
    return eng


def test_engine_layer_ids_and_drop_probabilities():
    eng = _cpu_engine(32, 'fp32')
    names = [b.name for b in eng.dspec.blocks]
    lay = eng.dropout_layers()
    assert list(lay) == ['enc1b', 'enc2b', 'enc3b', 'up3', 'up2', 'up1', 'up0']
    for n, (li, p) in lay.items():
        assert li == names.index(n) and p == (0.25 if n in ('enc1b', 'up0') else 0.5)
    ups = _cpu_engine(32, 'fp32', 'upsampling')
    nb = len(ups.dspec.blocks)
    assert [ups.dropout_layers()[n][0] for n in ('up3', 'up2', 'up1', 'up0')] == [nb, nb + 1, nb + 2, nb + 3]
    assert ups.dropout_layers()['enc2b'][0] == [b.name for b in ups.dspec.blocks].index('enc2b')


def test_engine_keep_masks_follow_the_seed_and_rank_rules():
    golden = 0x9E3779B97F4A7C15                         # the device seed after the first step (dcb_step_advance)
    B, H, W = 3, 16, 32
    m0 = dm.engine_keep_masks(_cpu_engine(32, 'fp32', step_seed=golden), B, H, W)
    assert dm.engine_keep_masks(_cpu_engine(32, 'fp32'), B, H, W, dropout=False) is None
    lay = _cpu_engine(32, 'fp32').dropout_layers()
    for name, (li, p) in lay.items():
        lvl = 3 if name in ('enc3b', 'up3') else 2 if name in ('enc2b', 'up2') else 1 if name in ('enc1b', 'up1') else 0
        c = 32 << lvl
        assert m0[name].shape == (B, c, H >> lvl, W >> lvl)
        want = dm.keep_scale(golden, li, m0[name].size, p).reshape(B, H >> lvl, W >> lvl, c).transpose(0, 3, 1, 2) > 0
        assert np.array_equal(m0[name], want), name
    # a second rank draws with seed rank * 0x9E3779B1 ^ step seed
    m1 = dm.engine_keep_masks(_cpu_engine(32, 'fp32', rank=1, step_seed=golden), B, H, W)
    li, p = lay['enc1b']
    want = dm.keep_scale(0x9E3779B1 ^ golden, li, m1['enc1b'].size, p).reshape(B, H >> 1, W >> 1, 64).transpose(0, 3, 1, 2) > 0
    assert np.array_equal(m1['enc1b'], want) and not np.array_equal(m1['enc1b'], m0['enc1b'])
    # the explicit step seed overrides the engine's state
    m2 = dm.engine_keep_masks(_cpu_engine(32, 'fp32'), B, H, W, step_seed=golden)
    assert all(np.array_equal(m2[k], m0[k]) for k in m0)


@pytest.mark.parametrize('nfb, mode, name', [(16, 'transpose', 'up0'), (8, 'transpose', 'enc1b'), (8, 'upsampling', 'up0')])
def test_engine_keep_masks_are_drawn_over_the_padded_width(nfb, mode, name):
    """bf16 pads every tensor narrower than 32 channels to 32 on the device (graph.padded_width): its mask is the crop of a
    32-channel draw, not a draw over the logical channels"""
    B, H, W, seed = 2, 8, 16, 0x0123456789ABCDEF
    eng = _cpu_engine(nfb, 'bf16', mode, step_seed=seed)
    masks = dm.engine_keep_masks(eng, B, H, W)
    li, p = eng.dropout_layers()[name]
    lvl = int(name[3] if name.startswith('enc') else name[2])
    h, w = H >> lvl, W >> lvl
    c = masks[name].shape[1]
    assert c == 16 and masks[name].shape == (B, c, h, w)
    full = dm.keep_scale(seed, li, B * h * w * 32, p).reshape(B, h, w, 32) > 0
    assert np.array_equal(masks[name], full[..., :c].transpose(0, 3, 1, 2))
    narrow = dm.keep_scale(seed, li, B * h * w * c, p).reshape(B, h, w, c) > 0
    assert not np.array_equal(masks[name], narrow.transpose(0, 3, 1, 2))
    # widths of 32 and more are not padded: the same draw as the fp32 check mode
    ref = dm.engine_keep_masks(_cpu_engine(nfb, 'fp32', mode, step_seed=seed), B, H, W)
    assert np.array_equal(masks['enc3b'], ref['enc3b'])
