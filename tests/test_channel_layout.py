"""The zero-padded device channel layout of the 16-bit precisions (engine/graph.py): the padded widths, the kernels'
width constraints, and the Keras <-> device weight and optimiser-state conversions."""
import numpy as np
import pytest

from deepcalcium.engine.graph import (GraphSpec, flat_layout, he_normal_weights, pack, pack_flat, padded_width, unpack,
                                      unpack_flat)

MODES = ('transpose', 'upsampling')


def _level_widths(spec):
    return [spec.by_name[n].cout for n in ('enc0b', 'enc1b', 'enc2b', 'enc3b', 'botb')]


@pytest.mark.parametrize('nfb, widths', [(8, [32, 32, 32, 64, 128]), (16, [32, 32, 64, 128, 256]),
                                         (24, [32, 64, 128, 256, 512]), (48, [64, 128, 256, 512, 1024])])
def test_padded_level_widths(nfb, widths):
    for mode in MODES:
        assert _level_widths(GraphSpec(nfb, upsampling_or_transpose=mode).device_spec('bf16')) == widths


@pytest.mark.parametrize('nfb', [32, 64])
@pytest.mark.parametrize('mode', MODES)
def test_nfb_32_and_64_map_to_themselves(nfb, mode):
    spec = GraphSpec(nfb, upsampling_or_transpose=mode)
    for precision in ('bf16', 'fp16'):
        d = spec.device_spec(precision)
        assert [(b.name, b.kind, b.cin, b.cout, b.level) for b in d.blocks] == \
               [(b.name, b.kind, b.cin, b.cout, b.level) for b in spec.blocks]
        assert d.cat_split == spec.cat_split
        assert flat_layout(d) == flat_layout(spec)
    assert all(padded_width(c) == c for c in (32, 64, 128, 256, 512, 1024))


def test_padded_width_values():
    assert [padded_width(c) for c in (1, 2, 3, 8, 16, 31, 32, 33, 48, 64, 65, 96, 192, 384, 768)] == \
           [32, 32, 32, 32, 32, 32, 32, 64, 64, 64, 128, 128, 256, 512, 1024]
    for c in (0, 1025):
        with pytest.raises(ValueError):
            padded_width(c)


@pytest.mark.parametrize('nfb', range(1, 65))
@pytest.mark.parametrize('mode', MODES)
def test_every_padded_width_meets_the_kernel_constraints(nfb, mode):
    d = GraphSpec(nfb, upsampling_or_transpose=mode).device_spec('bf16')
    assert d.by_name['enc0a'].cin == 1 and d.by_name['head'].cout == 2
    for blk in d.blocks:
        if blk.kind != 'head':
            c = blk.cout
            assert c % 32 == 0                                  # tensor-core convolutions: C0, C1, Cout multiples of 32
            assert c & (c - 1) == 0 and c <= 1024               # single-launch BatchNorm kernels
        if blk.name == 'enc0a':
            assert blk.cout in (8, 16, 32, 64)                  # first-layer conv (dcb_conv3x3_c1_fwd)
        if blk.name in d.cat_split:
            up = d.cat_split[blk.name]
            assert up % 32 == 0 and (blk.cin - up) % 32 == 0
        elif blk.name != 'enc0a':
            assert blk.cin % 32 == 0
    # the head reads dec0b's padded channels
    assert d.by_name['head'].cin == d.by_name['dec0b'].cout


def test_fp32_check_mode_stays_unpadded():
    spec = GraphSpec(16)
    assert spec.device_spec('fp32') is spec


def test_sixteen_bit_precisions_reject_nfb_65():
    for precision in ('bf16', 'fp16'):
        GraphSpec(64).device_spec(precision)
        with pytest.raises(ValueError, match='64'):
            GraphSpec(65).device_spec(precision)
    assert GraphSpec(65).device_spec('fp32').nfb == 65


def _random_weights(spec, seed):
    rng = np.random.default_rng(seed)
    return {k: rng.standard_normal(shp).astype(np.float32) for k, shp in spec.weight_shapes().items()}


@pytest.mark.parametrize('nfb', [1, 3, 8, 16, 24, 48])
@pytest.mark.parametrize('mode', MODES)
def test_pack_unpack_round_trip_is_bit_exact(nfb, mode):
    spec = GraphSpec(nfb, upsampling_or_transpose=mode)
    d = spec.device_spec('bf16')
    w = _random_weights(spec, nfb)
    p = pack(spec, d, w)
    shapes = d.weight_shapes()
    assert all(p[k].shape == tuple(shapes[k]) and p[k].dtype == np.float32 for k in w)
    back = unpack(spec, d, p)
    assert list(back.keys()) == list(w.keys())
    assert all(back[k].shape == w[k].shape and np.array_equal(back[k].view(np.uint32), w[k].view(np.uint32)) for k in w)


@pytest.mark.parametrize('nfb', [3, 16, 24])
@pytest.mark.parametrize('mode', MODES)
def test_padded_entries_hold_their_specified_values(nfb, mode):
    spec = GraphSpec(nfb, upsampling_or_transpose=mode)
    d = spec.device_spec('bf16')
    # real entries set to a value no padded entry takes: what is not NaN afterwards is padding
    w = {k: np.full(shp, np.nan, np.float32) for k, shp in spec.weight_shapes().items()}
    p = pack(spec, d, w)
    for k, a in p.items():
        pad = a[~np.isnan(a)]
        assert pad.size == a.size - w[k].size, k
        assert np.all(pad == (1. if k.endswith('/moving_var') else 0.)), k
    # concat layer: the skip channels start right after the padded up-path width
    name = 'dec0a'
    up_r, up_d = spec.cat_split[name], d.cat_split[name]
    k = p[name + '/kernel']
    co, skip = spec.by_name[name].cout, spec.by_name[name].cin - up_r
    assert np.isnan(k[:, :, :up_r, :co]).all() and not np.isnan(k[:, :, up_r:up_d]).any()
    assert np.isnan(k[:, :, up_d:up_d + skip, :co]).all() and not np.isnan(k[:, :, up_d + skip:]).any()
    assert not np.isnan(k[:, :, :, co:]).any()


@pytest.mark.parametrize('nfb', [1, 16, 24, 48])
@pytest.mark.parametrize('mode', MODES)
def test_optimizer_state_layout_round_trip(nfb, mode):
    spec = GraphSpec(nfb, upsampling_or_transpose=mode)
    d = spec.device_spec('bf16')
    slots, n, _ = flat_layout(spec)
    flat = np.zeros(n, np.float32)
    rng = np.random.default_rng(nfb)
    for k, (tr, off, shp) in slots.items():
        if tr:
            flat[off:off + int(np.prod(shp))] = rng.standard_normal(int(np.prod(shp)))
    dev = pack_flat(spec, d, flat)
    assert dev.shape == (flat_layout(d)[1],)
    assert np.array_equal(unpack_flat(spec, d, dev), flat)
    # the device vector is pack() of the per-array view: padded entries 0
    dslots = flat_layout(d)[0]
    w = {k: flat[off:off + int(np.prod(shp))].reshape(shp) for k, (tr, off, shp) in slots.items() if tr}
    for k, a in pack(spec, d, w).items():
        off = dslots[k][1]
        assert np.array_equal(dev[off:off + a.size], a.ravel()), k
    with pytest.raises(ValueError):
        pack_flat(spec, d, flat[:-4])


def test_he_normal_weights_pack_to_the_same_real_entries():
    spec = GraphSpec(16)
    d = spec.device_spec('fp16')
    w = he_normal_weights(spec, seed=3)
    p = pack(spec, d, w)
    assert np.array_equal(p['enc0a/kernel'][:, :, :, :16], w['enc0a/kernel'])
    assert np.array_equal(p['head/kernel'][:, :, :16], w['head/kernel'])
    assert np.array_equal(p['up0/kernel'][:, :, :16, :32], w['up0/kernel'])
