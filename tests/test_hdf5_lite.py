"""The pure-Python HDF5 subset (deepcalcium/utils/hdf5_lite.py) behind the reference's file formats (SURVEY N1 / N4):
pinned against a GENUINE libhdf5-written file - the MATLAB v7.3 test file that ships with scipy - and by write / read
round trips of the two layouts the reference uses (dataset schema of datasets/nf.py:39-44 and the Keras 2.0.6 model
layout of utils/keras_helpers.py:24-68).

tests/golden/testhdf5_7.4_GLNX86.mat and testdouble_7.4_GLNX86.mat are copies of scipy's io/matlab test data,
Copyright (c) 2001-2002 Enthought, Inc. 2003, SciPy Developers, under scipy's BSD 3-clause licence."""
import os

import numpy as np
import pytest

from deepcalcium.utils import hdf5_lite as h5


def test_reads_a_genuine_libhdf5_file(golden_dir):
    """superblock v0 behind a 512-byte user block, symbol-table root group, v1 object header, contiguous float64 dataset
    (layout message v2), fixed-length string attribute - written by MATLAB 7.4 through libhdf5 in 2008.  The expected
    values come from the SAME variable stored in MATLAB's own (non-HDF5) v7 format, read by scipy."""
    import scipy.io
    with h5.File(os.path.join(golden_dir, 'testhdf5_7.4_GLNX86.mat'), 'r') as f:
        assert f.keys() == ['testdouble'] and 'testdouble' in f and 'nope' not in f
        ds = f['testdouble']
        assert ds.shape == (9, 1) and ds.dtype == np.dtype('<f8')
        assert ds.attrs['MATLAB_class'] == b'double'
        got = ds[...]
    ref = scipy.io.loadmat(os.path.join(golden_dir, 'testdouble_7.4_GLNX86.mat'))['testdouble']
    assert np.array_equal(got.ravel(), ref.ravel())
    assert np.allclose(got.ravel(), np.linspace(0, 2 * np.pi, 9))


def test_rejects_non_hdf5_and_new_format(tmp_path):
    p = tmp_path / 'x.hdf5'
    p.write_bytes(b'not hdf5' * 100)
    with pytest.raises(h5.Hdf5Error):
        h5.File(str(p), 'r')
    p.write_bytes(h5.SIGNATURE + bytes([2]) + b'\x00' * 100)
    with pytest.raises(h5.Hdf5Error, match='superblock version 2'):
        h5.File(str(p), 'r')


def test_write_read_round_trip_of_every_supported_type(tmp_path):
    rng = np.random.default_rng(0)
    arrays = {'f32': rng.standard_normal((3, 4, 5)).astype(np.float32), 'f16': rng.standard_normal((7, 2)).astype(np.float16),
              'f64': rng.standard_normal(11), 'i16': rng.integers(-3000, 3000, (4, 6)).astype(np.int16),
              'i8': rng.integers(-100, 100, (2, 3, 4)).astype(np.int8), 'u8': rng.integers(0, 255, 9).astype(np.uint8),
              'i64': rng.integers(-2 ** 40, 2 ** 40, 5), 'scalar': np.float32(3.5), 'empty': np.zeros((0, 4), np.float32)}
    path = str(tmp_path / 'rt.hdf5')
    with h5.File(path, 'w') as f:
        f.attrs['name'] = 'neurofinder.00.00'
        f.attrs['count'] = np.int64(7)
        f.attrs['names'] = np.array([b'alpha', b'be', b'gamma_delta'])
        g = f.create_group('a/b')
        for k, v in arrays.items():
            d = g.create_dataset(k, data=v)
            d.attrs['unit'] = b'px'
        many = f.create_group('many')                       # more links than one symbol-table node holds
        for i in range(150):
            many.create_dataset('d%03d' % i, data=np.full(3, i, np.int32))
    with h5.File(path, 'r') as f:
        assert f.attrs['name'] == b'neurofinder.00.00' and int(f.attrs['count']) == 7
        assert [bytes(x) for x in f.attrs['names']] == [b'alpha', b'be', b'gamma_delta']
        assert f.keys() == ['a', 'many'] and f['a'].keys() == ['b']
        for k, v in arrays.items():
            d = f['a/b/' + k]
            assert d.dtype == np.asarray(v).dtype and tuple(d.shape) == np.asarray(v).shape, k
            assert np.array_equal(d[...], v), k
            assert d.attrs['unit'] == b'px'
        assert len(f['many'].keys()) == 150
        for i in (0, 31, 32, 99, 149):
            assert np.array_equal(f['many/d%03d' % i][...], np.full(3, i, np.int32))
        assert np.array_equal(f['a/b/f32'][1, :, 2], arrays['f32'][1, :, 2])


def test_dataset_schema_of_the_reference(tmp_path):
    """datasets/nf.py:39-44,113-125: series/mean float16, series/max int16, masks/raw int8, masks/max int8, attr name"""
    from deepcalcium.datasets.nf import make_dataset, open_dataset
    rng = np.random.default_rng(1)
    mean = rng.random((40, 56)).astype(np.float32) * 300
    mx = mean * 2 + 70000 * (rng.random(mean.shape) < 0.01)          # a few values beyond int16: saturate like HDF5 does
    masks = (rng.random((5, 40, 56)) < 0.05).astype(np.int8)
    path = make_dataset(str(tmp_path / 'dataset.hdf5'), 'neurofinder.01.00', mean=mean, mx=mx, masks=masks)
    with h5.File(path, 'r') as f:
        assert f.attrs['name'] == b'neurofinder.01.00'
        assert f['series/mean'].dtype == np.float16 and f['series/max'].dtype == np.int16
        assert f['masks/raw'].dtype == np.int8 and f['masks/raw'].shape == (5, 40, 56)
    ds = open_dataset(path)
    assert ds['name'] == 'neurofinder.01.00'
    assert np.array_equal(ds['series/mean'], mean.astype(np.float16))
    assert ds['series/max'].max() == 32767 and np.array_equal(ds['masks/max'], masks.max(0))


@pytest.mark.parametrize('mode', ['transpose', 'upsampling'])
def test_keras_model_layout_round_trip(tmp_path, mode):
    """utils/keras_helpers.py:24-68 / unet_2d_summary.py:423-424: model_weights/<layer>/<layer>/<weight>:0 datasets, layer_names
    and weight_names attributes in Keras' layer order; 134 arrays for the default graph."""
    from deepcalcium.engine.graph import GraphSpec, he_normal_weights
    from deepcalcium.utils.keras_hdf5 import write_keras_model, read_keras_weights, keras_layer_names, is_hdf5
    spec = GraphSpec(32, 0.2, mode)
    w = he_normal_weights(spec, seed=5)
    rng = np.random.default_rng(5)
    for k in w:
        w[k] = (w[k] + 0.01 * rng.standard_normal(w[k].shape)).astype(np.float32)
    path = write_keras_model(str(tmp_path / 'model.hdf5'), spec, w, (96, 96), optimizer={'lr': 0.002}, loss='dice_loss')
    assert is_hdf5(path)
    with h5.File(path, 'r') as f:
        assert f.attrs['keras_version'] == b'2.0.6'
        mw = f['model_weights']
        names = [bytes(x).decode() for x in mw.attrs['layer_names']]
        assert names == [n for n, _ in keras_layer_names(spec)]
        assert names[2] == 'conv2d_1' and names[-2] == 'conv2d_19' and names[-1] == 'lambda_2'
        assert [bytes(x) for x in mw['conv2d_1'].attrs['weight_names']] == [b'conv2d_1/kernel:0', b'conv2d_1/bias:0']
        assert mw['conv2d_1/conv2d_1/kernel:0'].shape == (3, 3, 1, 32)
        assert [bytes(x) for x in mw['batch_normalization_1'].attrs['weight_names']][3] == b'batch_normalization_1/moving_variance:0'
        assert len(mw['activation_1'].attrs['weight_names']) == 0
        if mode == 'transpose':
            assert mw['conv2d_transpose_1/conv2d_transpose_1/kernel:0'].shape == (2, 2, 256, 512)
    spec2, w2, info = read_keras_weights(path)
    assert (spec2.nfb, spec2.up_mode, spec2.drp) == (32, mode, 0.2)
    assert list(w2.keys()) == list(w.keys()) and all(np.array_equal(w[k], w2[k]) for k in w)
    assert len(w2) == (134 if mode == 'transpose' else 110)
    assert info['training_config']['loss'] == 'dice_loss'
