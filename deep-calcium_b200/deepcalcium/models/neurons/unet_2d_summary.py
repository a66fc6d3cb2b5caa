"""UNet2DS wrapper with the reference's Python surface
(deepcalcium/models/neurons/unet_2d_summary.py): ``unet``, ``UNet2DSummary.fit / predict`` plus an
``evaluate`` method that is the reference CLI's evaluation() (examples/neurons/unet2ds_nf.py:47-64).

No Keras / TensorFlow: the model object returned by ``unet()`` drives hand-written sm_100a kernels
through the C ABI (include/dcb200.h).  There is no CPU fallback.
"""
from __future__ import division, print_function

import csv
import json
import logging
import os
import pickle
from os import path
from time import time

import numpy as np

from ...engine.graph import GraphSpec, MAX_NFB_16BIT, flat_layout, weights_to_list, list_to_weights, he_normal_weights
from ...utils.runtime import funcname
from ...utils import neurons as _un
from ...utils.neurons import (F1, prec, reca, dice, dicesq, dice_loss, dicesq_loss, posyt, posyp,
                              weighted_binary_crossentropy, binary_crossentropy)
from ...datasets.nf import open_dataset, nf_mask_metrics_device, summarize_masks_device

MODEL_URL_LATEST = 'https://github.com/alexklibisz/deep-calcium/releases/download/v0.0.1-weights/unet2ds_model.hdf5'
METRIC_NAMES = ['loss', 'F1', 'prec', 'reca', 'dice', 'dicesq', 'posyt', 'posyp']   # unet_2d_summary.py:398-399


class Adam(object):
    """Stand-in for keras.optimizers.Adam (Keras 2.0.6 update rule, unet_2d_summary.py:335)."""

    def __init__(self, lr=0.001, beta_1=0.9, beta_2=0.999, epsilon=1e-8):
        self.lr, self.beta_1, self.beta_2, self.epsilon = float(lr), float(beta_1), float(beta_2), float(epsilon)

    def get_config(self):
        return dict(lr=self.lr, beta_1=self.beta_1, beta_2=self.beta_2, epsilon=self.epsilon)


class UNetModel(object):
    """What ``unet()`` returns: the subset of the Keras ``Model`` surface the reference uses
    (input_shape :76,570; predict :87,588,592; get_weights / set_weights :69; train_on_batch via
    fit_generator :429)."""

    def __init__(self, window_shape, spec, precision=None, seed=None):
        from ...engine.unet_engine import UNetEngine
        assert len(window_shape) == 2
        self.window_shape = tuple(int(v) for v in window_shape)
        self.spec = spec
        precision = precision or _default_precision(spec, True)   # inference-only loads use 'fp16' (see load_model_...)
        self.engine = UNetEngine(spec, precision=precision)
        self.engine.set_weights_dict(he_normal_weights(spec, seed))
        self.optimizer = Adam(0.002)
        self.loss = 'binary_crossentropy'
        self.dropout = True

    @property
    def input_shape(self):
        return (None,) + self.window_shape

    def get_weights(self):
        return weights_to_list(self.spec, self.engine.get_weights_dict())

    def set_weights(self, weights):
        self.engine.set_weights_dict(list_to_weights(self.spec, weights))

    def compile(self, optimizer=None, loss='binary_crossentropy', metrics=None):
        self.optimizer = optimizer or Adam(0.002)
        self.loss = loss if isinstance(loss, str) else loss.__name__
        if self.loss not in _un.LOSS_IDS:
            raise ValueError('unknown loss %r' % (loss,))
        self.engine.reset_optimizer()

    def predict(self, x, batch_size=None):
        """x: [N,H,W] array -> float32 [N,H,W] probabilities (softmax channel -1)."""
        import torch
        x = np.ascontiguousarray(np.asarray(x, dtype=np.float32))
        if x.ndim != 3:
            raise ValueError('predict expects [N,H,W], got %s' % (x.shape,))
        prob, _ = self.engine.infer(torch.from_numpy(x).cuda())
        return prob.cpu().numpy()

    def predict_logits(self, x):
        import torch
        x = np.ascontiguousarray(np.asarray(x, dtype=np.float32))
        _, logit = self.engine.infer(torch.from_numpy(x).cuda())
        return logit.cpu().numpy()

    def train_on_batch(self, x, y):
        """One optimiser step; returns [loss, F1, prec, reca, dice, dicesq, posyt, posyp]."""
        import torch
        if not (torch.is_tensor(x) and x.is_cuda):       # host batches (reference-style generators) are uploaded here
            x = torch.from_numpy(np.ascontiguousarray(np.asarray(x, dtype=np.float32))).cuda()
            y = torch.from_numpy(np.ascontiguousarray(np.asarray(y, dtype=np.uint8))).cuda()
        o = self.optimizer
        m = self.engine.train_step(x, y, loss=self.loss, lr=o.lr, dropout=self.dropout, beta1=o.beta_1,
                                   beta2=o.beta_2, eps=o.epsilon)
        return m.cpu().numpy().tolist()

    # ---- persistence.  *.hdf5 / *.h5: the Keras-2.0.6 model layout the reference writes (utils/keras_hdf5.py: readable by
    # Keras' load_weights and by this package); anything else: an .npz container with the same arrays
    def save(self, filepath, include_optimizer=True):
        e = self.engine
        w = e.get_weights_dict()
        extra = {}
        if include_optimizer:         # the unpadded layout of every precision: a checkpoint loads into any of them
            extra = dict(e.get_optimizer_state())
        if filepath.endswith(('.hdf5', '.h5')):
            from ...utils.keras_hdf5 import write_keras_model
            write_keras_model(filepath, self.spec, w, self.window_shape, optimizer=self.optimizer.get_config(), loss=self.loss,
                              extra_attrs={'deepcalcium_iteration': np.int64(e.iteration)}, extra_datasets=extra)
            return
        cfg = dict(format='deepcalcium-b200-v1', nb_filters_base=self.spec.nfb, prop_dropout_base=self.spec.drp,
                   upsampling_or_transpose=self.spec.up_mode, window_shape=list(self.window_shape),
                   optimizer=self.optimizer.get_config(), loss=self.loss, iteration=int(e.iteration),
                   weight_keys=list(w.keys()))
        arrays = {'w%03d' % i: v for i, v in enumerate(w.values())}
        arrays.update(extra)
        arrays['config'] = np.asarray(json.dumps(cfg))
        with open(filepath, 'wb') as fp:
            np.savez(fp, **arrays)

    def load_weights(self, filepath):
        """keras.Model.load_weights for a Keras-layout HDF5 file of the same graph"""
        from ...utils.keras_hdf5 import read_keras_weights
        spec, w, _ = read_keras_weights(filepath)
        if (spec.nfb, spec.up_mode) != (self.spec.nfb, self.spec.up_mode):
            raise ValueError('%s holds a %d-filter %s graph, this model is %d / %s'
                             % (filepath, spec.nfb, spec.up_mode, self.spec.nfb, self.spec.up_mode))
        self.engine.set_weights_dict(w)


def _default_precision(spec, trainable):
    # predict() loads with trainable=False: inference only -> fp16 activations (same tensor-core rate as bf16, 8x smaller
    # logit error: meets the 1e-2 tolerance); a model that will be trained is bf16.  The 16-bit modes run every
    # nb_filters_base up to 64 (narrower ones on zero-padded channels); wider networks run in the fp32 check mode.
    return 'fp32' if spec.nfb > MAX_NFB_16BIT else ('bf16' if trainable else 'fp16')


def load_model_with_new_input_shape(model_path, input_shape, compile=True, precision=None, trainable=True, **kwargs):
    """Counterpart of deepcalcium/utils/keras_helpers.py:24-68: the graph is fully convolutional, so the same weights
    simply run at another window size (no file rewriting).  Reads Keras-2.x HDF5 model files (the reference's
    checkpoints, the released unet2ds_model.hdf5) and this package's .npz containers."""
    from ...utils.keras_hdf5 import is_hdf5, read_keras_weights, read_extra
    if is_hdf5(model_path):
        spec, w, info = read_keras_weights(model_path)
        model = UNetModel(tuple(input_shape), spec, precision=precision or _default_precision(spec, trainable))
        model.engine.set_weights_dict(w)
        tc = info.get('training_config') or {}
        oc = (tc.get('optimizer_config') or {}).get('config') or {}
        if oc:
            model.optimizer = Adam(lr=oc.get('lr', 0.002), beta_1=oc.get('beta_1', 0.9), beta_2=oc.get('beta_2', 0.999),
                                   epsilon=oc.get('epsilon', 1e-8))
        if tc.get('loss') in _un.LOSS_IDS:
            model.loss = tc['loss']
        if compile:
            ex = read_extra(model_path, ('adam_m', 'adam_v', 'step_state'))
            if len(ex) == 3 and ex['adam_m'].shape == (flat_layout(spec)[1],):
                model.engine.set_optimizer_state(ex['adam_m'], ex['adam_v'], ex['step_state'])
        return model
    with np.load(model_path, allow_pickle=False) as z:
        cfg = json.loads(str(z['config']))
        if cfg.get('format') != 'deepcalcium-b200-v1':
            raise ValueError('%s is not a deepcalcium-b200 model file' % model_path)
        spec = GraphSpec(cfg['nb_filters_base'], cfg['prop_dropout_base'], cfg['upsampling_or_transpose'])
        model = UNetModel(tuple(input_shape), spec, precision=precision or _default_precision(spec, trainable))
        model.engine.set_weights_dict({k: z['w%03d' % i] for i, k in enumerate(cfg['weight_keys'])})
        model.optimizer = Adam(**cfg['optimizer'])
        model.loss = cfg['loss']
        if compile and 'adam_m' in z.files:
            model.engine.set_optimizer_state(z['adam_m'], z['adam_v'], z['step_state'])
            model.engine.iteration = int(cfg['iteration'])
    return model


def unet(window_shape=(128, 128), nb_filters_base=32, conv_kernel_init='he_normal',
         prop_dropout_base=0.25, upsampling_or_transpose='transpose', precision=None, seed=None):
    """Same arguments as the reference's unet() (unet_2d_summary.py:123-124).  ``precision`` selects 'bf16' (tcgen05
    kernels, default: trainable), 'fp16' (same kernels with fp16 storage, inference only) or 'fp32' (CUDA-core check mode).
    The 16-bit modes take nb_filters_base up to 64 (ValueError above that); wider networks default to 'fp32'."""
    assert len(window_shape) == 2 and window_shape[0] == window_shape[1]
    if conv_kernel_init != 'he_normal':
        raise NotImplementedError("only conv_kernel_init='he_normal' (the reference default) is built")
    mode = 'transpose' if upsampling_or_transpose == 'transpose' else 'upsampling'
    return UNetModel(window_shape, GraphSpec(nb_filters_base, prop_dropout_base, mode), precision=precision, seed=seed)


# ------------------------------------------------------------------ default summary functions
def _summarize_series(dspath):
    """unet_2d_summary.py:227-241: series/mean -> float32 -> (x - mean) / std, on the GPU."""
    import torch
    from ...engine import ops
    ds = open_dataset(dspath, keys=('series/mean',))
    summ = torch.from_numpy(np.ascontiguousarray(ds['series/mean'].astype(np.float32))).cuda()
    out = torch.empty_like(summ)
    ops.standardize(summ, out)
    return out.cpu().numpy()


def _summarize_mask(dspath):
    """unet_2d_summary.py:244-291: flatten the per-neuron masks; drop pixels claimed by more than one
    neuron, then drop any 3x3 neighbourhood that still touches two different neurons (same visiting
    order as the reference: first-seen order of the (y,x) keys).  Runs on the GPU (summarize_masks_device);
    returns float64 [H, W] like the reference."""
    import torch
    msks = open_dataset(dspath, keys=('masks/raw',))['masks/raw']
    if msks.dtype.itemsize != 1 or msks.dtype.kind not in 'biu':
        msks = msks == 1                       # the device takes one-byte planes; "== 1" is the only test applied
    out = summarize_masks_device(torch.from_numpy(np.ascontiguousarray(msks)).cuda())
    return out.cpu().numpy().astype(np.float64)


def _name_dataset(dspath):
    return open_dataset(dspath, keys=())['name']


def _pixel_scores(m, mp):
    """Pixel-level precision / recall / F1 (utils/neurons.py:32-50 on hard masks); kept as a cheap diagnostic next to
    the region-level nf_mask_metrics the reference reports."""
    m, mp = np.asarray(m, np.float64), np.asarray(mp, np.float64)
    return float(prec(m, mp)), float(reca(m, mp)), float(F1(m, mp))


class UNet2DSummary(object):
    """Same constructor and methods as the reference class (unet_2d_summary.py:301-625)."""

    def __init__(self, cpdir=None, dataset_name_func=_name_dataset, series_summary_func=_summarize_series,
                 mask_summary_func=_summarize_mask, net_builder_func=unet):
        if cpdir is None:
            from ...utils.config import CHECKPOINTS_DIR
            cpdir = '%s/neurons_unet2ds' % CHECKPOINTS_DIR
        self.cpdir = cpdir
        self.dataset_name_func = dataset_name_func
        self.series_summary_func = series_summary_func
        self.mask_summary_func = mask_summary_func
        self.net_builder_func = net_builder_func
        os.makedirs(self.cpdir, exist_ok=True)
        cobj = [F1, prec, reca, dice, dicesq, posyt, posyp, dice_loss, dicesq_loss]
        self.custom_objects = {x.__name__: x for x in cobj}

    # ------------------------------------------------------------------ fit
    def fit(self, dataset_paths, model_path=None, proceed=False, shape_trn=(96, 96), shape_val=(512, 512),
            batch_size_trn=32, batch_size_val=1, nb_steps_trn=200, nb_epochs=20, prop_trn=0.75, prop_val=0.25,
            keras_callbacks=[], optimizer=None, loss='binary_crossentropy'):
        """unet_2d_summary.py:333-432.  Returns (history dict, path of the last checkpoint)."""
        logger = logging.getLogger(funcname())
        assert len(shape_trn) == 2
        assert len(shape_val) == 2
        assert shape_trn[0] == shape_trn[1]
        assert shape_val[0] == shape_val[1]
        assert 0 < prop_trn < 1
        assert 0 < prop_val < 1
        assert not (proceed and not model_path)
        losses = ('binary_crossentropy', 'weighted_binary_crossentropy', 'dice_loss', 'dicesq_loss')
        loss_name = loss if isinstance(loss, str) else getattr(loss, '__name__', None)
        assert loss_name in losses
        optimizer = optimizer or Adam(0.002)

        if model_path:
            model = load_model_with_new_input_shape(model_path, shape_trn, compile=proceed)
        else:
            model = self.net_builder_func(shape_trn)
        if not proceed:
            model.compile(optimizer=optimizer, loss=loss_name,
                          metrics=[F1, prec, reca, dice, dicesq, posyt, posyp])

        names = [self.dataset_name_func(dsp) for dsp in dataset_paths]
        S_summ = [self.series_summary_func(dsp) for dsp in dataset_paths]
        M_summ = [self.mask_summary_func(dsp) for dsp in dataset_paths]
        ycval = [(s.shape[0] - int(s.shape[0] * prop_val), s.shape[0]) for s in S_summ]
        yctrn = [(0, int(s.shape[0] * prop_trn)) for s in S_summ]
        # the reference's _batch_gen (:434-530) with the same global-numpy RNG stream and the same crops; the pixel work
        # (slice, zero fill, flips / rot90s) runs on the GPU and the batch never visits the host
        gen_trn = self._batch_gen(S_summ, M_summ, names, yctrn, batch_size_trn, nb_steps_trn, shape_trn, 15,
                                  device=model.engine.dev)
        val = self._validation_data(S_summ, M_summ, model.engine.dev)

        for cb in keras_callbacks:               # Keras calls these before the first epoch
            if hasattr(cb, 'set_model'):
                cb.set_model(model)
            if hasattr(cb, 'on_train_begin'):
                cb.on_train_begin({})
        tic = int(time())
        csv_path = '%s/%d_metrics.csv' % (self.cpdir, tic)
        history = {}
        best_f1, since_best, last_path = -np.inf, 0, None
        for epoch in range(nb_epochs):
            acc = np.zeros(len(METRIC_NAMES))
            for _ in range(nb_steps_trn):
                xb, yb = next(gen_trn)
                acc += np.asarray(model.train_on_batch(xb, yb))
            logs = dict(zip(METRIC_NAMES, (acc / nb_steps_trn).tolist()))
            logs.update(self._validate(model, S_summ, M_summ, names, ycval, shape_val, epoch, val))
            logs['lr'] = model.optimizer.lr
            # ModelCheckpoint every epoch (:423-424)
            last_path = '%s/%d_model_%02d_%.3f.hdf5' % (self.cpdir, tic, epoch, logs['val_nf_f1_mean'])
            model.save(last_path)
            # ReduceLROnPlateau(monitor='F1', factor=0.5, patience=5, min_lr=1e-4, mode='max') (:425-426)
            # Keras 2.0.6 order: the patience test comes BEFORE the wait counter is incremented, so the rate is halved
            # on the 6th non-improving epoch; after a reduction the counter restarts at 1 (wait = 0, then += 1)
            if logs['F1'] > best_f1 + 1e-4:
                best_f1, since_best = logs['F1'], 0
            else:
                if since_best >= 5:
                    if model.optimizer.lr > 1e-4 + 1e-4 * 1e-4:
                        model.optimizer.lr = max(model.optimizer.lr * 0.5, 1e-4)
                        since_best = 0
                since_best += 1
            for cb in keras_callbacks:
                cb.on_epoch_end(epoch, logs)
            for k, v in logs.items():
                history.setdefault(k, []).append(v)
            with open(csv_path, 'w') as fp:          # CSVLogger (:420)
                wr = csv.writer(fp)
                keys = sorted(history.keys())
                wr.writerow(['epoch'] + keys)
                for i in range(epoch + 1):
                    wr.writerow([i] + [history[k][i] for k in keys])
            logger.info('epoch %d: %s' % (epoch, ' '.join('%s=%.4f' % kv for kv in sorted(logs.items()))))
        return history, last_path

    # The six orientations of _ValidationMetricsCB (:62-120): f_k = identity, np.fliplr, np.flipud, np.rot90 k = 1, 2, 3.
    # _VAL_SRC[k](H, W, a, b) = the pixel (i, j) of an H x W image that f_k puts at (a, b); _VAL_DST is its inverse.
    _VAL_SRC = (lambda H, W, a, b: (a, b), lambda H, W, a, b: (a, W - 1 - b), lambda H, W, a, b: (H - 1 - a, b),
                lambda H, W, a, b: (b, W - 1 - a), lambda H, W, a, b: (H - 1 - a, W - 1 - b),
                lambda H, W, a, b: (H - 1 - b, a))
    _VAL_DST = (lambda H, W, y, x: (y, x), lambda H, W, y, x: (y, W - 1 - x), lambda H, W, y, x: (H - 1 - y, x),
                lambda H, W, y, x: (W - 1 - x, y), lambda H, W, y, x: (H - 1 - y, W - 1 - x),
                lambda H, W, y, x: (x, H - 1 - y))

    @classmethod
    def _val_box(cls, shape, y0, y1, k):
        """(a0, a1, b0, b1): the smallest and largest row and column that the validation rows [y0, y1) of an image of
        `shape` occupy after orientation k - the reference's np.where(f(vm) == 1) box (scored as [a0:a1, b0:b1], the
        exclusive max() end kept), taken from the corners of the band"""
        H, W = shape
        if not (0 <= y0 < y1 <= H) or W == 0:
            raise ValueError('validation rows [%d, %d) are empty in a %d x %d image' % (y0, y1, H, W))
        pts = [cls._VAL_DST[k](H, W, y, x) for y in (y0, y1 - 1) for x in (0, W - 1)]
        return min(p[0] for p in pts), max(p[0] for p in pts), min(p[1] for p in pts), max(p[1] for p in pts)

    @staticmethod
    def _validation_data(S_summ, M_summ, dev):
        """the summary images (fp32) and truth masks (m != 0 as uint8) on the device, uploaded once per fit"""
        import torch
        return [(torch.from_numpy(np.ascontiguousarray(s, dtype=np.float32)).to(dev),
                 torch.from_numpy(np.ascontiguousarray(np.asarray(m) != 0, dtype=np.uint8)).to(dev))
                for s, m in zip(S_summ, M_summ)]

    def _validate(self, model, S_summ, M_summ, names, y_coords, shape_val, epoch, val=None):
        """_ValidationMetricsCB.on_epoch_end (:62-120): six orientations of every dataset at the validation window, scored
        inside the validation rows with the Neurofinder region matching (nf_mask_metrics).  Runs on the device: each
        orientation is reflect-padded to the window by ops.orient_pad and predicted at batch 1 as the reference does
        (images larger than the window: the identity transform over overlapping tiles); the truth masks are strided views
        of the uploaded masks, and all datasets x orientations are scored in one nf_metrics_from_table call.  `val`:
        _validation_data(S_summ, M_summ) (built here when not given)."""
        import torch
        from ...engine import ops
        from ...datasets.nf import nf_metrics_from_table
        dev = model.engine.dev
        if val is None:
            val = self._validation_data(S_summ, M_summ, dev)
        hw, ww = shape_val
        win = torch.empty(hw, ww, dtype=torch.float32, device=dev)
        preds, rows = [], []
        with torch.cuda.device(dev):
            for (s, m), (y0, y1) in zip(val, y_coords):
                H, W = s.shape
                for k in range(6):
                    hf, wf = (W, H) if k in (3, 5) else (H, W)
                    a0, a1, b0, b1 = self._val_box((H, W), y0, y1, k)
                    if hf <= hw and wf <= ww:
                        ops.orient_pad(s, k, win)
                        mp, kind = model.engine.infer(win[None])[0][0].clone(), 1
                    else:
                        fs = torch.empty(hf, wf, dtype=torch.float32, device=dev)
                        ops.orient_pad(s, k, fs)
                        mp, kind = model.engine.predict_tiled(fs, augmentation=False)[1].clone(), 2
                    preds.append(mp)
                    # truth: f_k(m)[a0:a1, b0:b1] as a signed-stride view of m (uint8, row-major H x W)
                    src = self._VAL_SRC[k]
                    off = [i * W + j for i, j in (src(H, W, a0, b0), src(H, W, a0 + 1, b0), src(H, W, a0, b0 + 1))]
                    rows.append([m.data_ptr() + off[0], a1 - a0, b1 - b0, off[1] - off[0], off[2] - off[0], 0, 0, 0])
                    rows.append([mp.data_ptr() + (a0 * mp.stride(0) + b0) * mp.element_size(), a1 - a0, b1 - b0,
                                 mp.stride(0), 1, kind, 0, 0])
            scores = nf_metrics_from_table(np.asarray(rows, dtype=np.int64), dev)
        pp = [sc[0] for sc in scores]
        rr = [sc[1] for sc in scores]
        ff = [sc[4] for sc in scores]
        eps = 1e-4 * epoch if epoch else 0
        return {'val_nf_f1_mean': float(np.mean(ff) + eps), 'val_nf_f1_median': float(np.median(ff) + eps),
                'val_nf_f1_min': float(np.min(ff) + eps), 'val_nf_f1_adj': float(np.mean(ff) * np.min(ff) + eps),
                'val_nf_prec': float(np.mean(pp)), 'val_nf_reca': float(np.mean(rr))}

    # D4 elements of the sampler's augment_funcs as index maps on an n x n window: out[i, j] = a[M @ (i, j) + t]
    @staticmethod
    def _aug_maps(n):
        return [((1, 0, 0, 1), (0, 0)),              # identity
                ((1, 0, 0, -1), (0, n - 1)),         # a[:, ::-1]
                ((-1, 0, 0, 1), (n - 1, 0)),         # a[::-1, :]
                ((0, 1, -1, 0), (0, n - 1)),         # np.rot90(a, 1): out[i, j] = a[j, n-1-i]
                ((-1, 0, 0, -1), (n - 1, n - 1)),    # np.rot90(a, 2)
                ((0, -1, 1, 0), (n - 1, 0))]         # np.rot90(a, 3): out[i, j] = a[n-1-j, i]

    def _crop_descriptors(self, S_summ, M_summ, names, y_coords, batch_size, nb_steps, window_shape,
                          nb_max_augment=0, scores_path=None):
        """The random half of the reference's _batch_gen (unet_2d_summary.py:434-530): yields int32 [batch, 12] crop
        descriptors {dataset, y0, x0, valid rows, valid cols, m00, m01, m10, m11, t0, t1, 0} drawing from the global numpy
        RNG in exactly the order the reference does (dataset, neuron, row jitter, column jitter, augmentation count,
        augmentation picks), so the same seed gives the same crops (tests/test_sampler.py against oracle/sampler.py)."""
        rng = np.random
        hw, ww = window_shape
        assert hw == ww, 'the flips / rotations are composed on a square window'
        maps = self._aug_maps(hw)
        nb_yields = 0
        neuron_locs = []
        for ds_idx, m in enumerate(M_summ):
            ymin, ymax = y_coords[ds_idx]
            neuron_locs.append(list(zip(*np.where(m[ymin:ymax, :] == 1))))
        ds_idxs = np.arange(len(S_summ))
        ds_idxp = np.ones((len(ds_idxs))) / len(ds_idxs)
        while True:
            if scores_path and os.path.exists(scores_path) and (nb_yields - 1) % nb_steps == 0:
                with open(scores_path, 'rb') as fp:
                    names_to_scores = pickle.load(fp)
                ds_idxp = np.array([1 - np.mean(names_to_scores[n]) for n in names])
                ds_idxp /= np.sum(ds_idxp)
            desc = np.zeros((batch_size, 12), dtype=np.int32)
            for b_idx in range(batch_size):
                ds_idx = rng.choice(np.arange(len(S_summ)), p=ds_idxp)
                hs, ws = S_summ[ds_idx].shape
                ymin, ymax = y_coords[ds_idx]
                cy, cx = neuron_locs[ds_idx][rng.randint(0, len(neuron_locs[ds_idx]))]
                cy = min(max(ymin, cy + rng.randint(-5, 5)), ymax)
                cx = min(max(0, cx + rng.randint(-5, 5)), ws)
                y0 = max(ymin, int(cy - (hw / 2)))
                y1 = min(y0 + hw, ymax)
                x0 = max(0, int(cx - (ww / 2)))
                x1 = min(x0 + ww, ws)
                nb_augment = rng.randint(0, nb_max_augment + 1)
                M, t = (1, 0, 0, 1), (0, 0)
                for k in rng.choice(len(maps), nb_augment):        # same draw as rng.choice(augment_funcs, nb_augment)
                    (a, b, c, d), (t0, t1) = maps[int(k)]
                    # cur = aug(prev): cur[p] = prev[Mk p + tk] = a[M (Mk p + tk) + t]
                    t = (M[0] * t0 + M[1] * t1 + t[0], M[2] * t0 + M[3] * t1 + t[1])
                    M = (M[0] * a + M[1] * c, M[0] * b + M[1] * d, M[2] * a + M[3] * c, M[2] * b + M[3] * d)
                desc[b_idx] = (ds_idx, y0, x0, y1 - y0, x1 - x0, M[0], M[1], M[2], M[3], t[0], t[1], 0)
            nb_yields += 1
            yield desc

    @staticmethod
    def _apply_descriptors_host(S_summ, M_summ, desc, n):
        """numpy statement of dcb_crop_batch (used by the CPU tests to pin the descriptors against the host sampler of oracle/)"""
        B = desc.shape[0]
        xs = np.zeros((B, n, n), np.float32); ys = np.zeros((B, n, n), np.uint8)
        ii, jj = np.meshgrid(np.arange(n), np.arange(n), indexing='ij')
        for b in range(B):
            ds, y0, x0, vh, vw, m00, m01, m10, m11, t0, t1, _ = (int(v) for v in desc[b])
            wi, wj = m00 * ii + m01 * jj + t0, m10 * ii + m11 * jj + t1
            ok = (wi >= 0) & (wi < vh) & (wj >= 0) & (wj < vw)
            xs[b][ok] = S_summ[ds][y0 + wi[ok], x0 + wj[ok]]
            ys[b][ok] = M_summ[ds][y0 + wi[ok], x0 + wj[ok]]
        return xs, ys

    def _batch_gen(self, S_summ, M_summ, names, y_coords, batch_size, nb_steps, window_shape,
                   nb_max_augment=0, scores_path=None, device=None):
        """The reference's crop sampler (unet_2d_summary.py:434-530) with the pixel work on the GPU (dcb_crop_batch):
        yields (x, y) CUDA tensors.  The summary images and masks are uploaded once; per batch only the [batch, 12]
        int32 descriptors cross PCIe."""
        import torch
        from ...engine import ops
        dev = device if device is not None else torch.device('cuda', torch.cuda.current_device())
        imgs = [torch.from_numpy(np.ascontiguousarray(np.asarray(s, dtype=np.float32))).to(dev) for s in S_summ]
        msks = [torch.from_numpy(np.ascontiguousarray(np.asarray(m, dtype=np.uint8))).to(dev) for m in M_summ]
        iptr = torch.tensor([t.data_ptr() for t in imgs], dtype=torch.int64, device=dev)
        mptr = torch.tensor([t.data_ptr() for t in msks], dtype=torch.int64, device=dev)
        wid = torch.tensor([t.shape[1] for t in imgs], dtype=torch.int32, device=dev)
        n = window_shape[0]
        xb = torch.empty(batch_size, n, n, dtype=torch.float32, device=dev)
        yb = torch.empty(batch_size, n, n, dtype=torch.uint8, device=dev)
        hdesc = torch.empty(batch_size, 12, dtype=torch.int32).pin_memory()
        ddesc = torch.empty(batch_size, 12, dtype=torch.int32, device=dev)
        for desc in self._crop_descriptors(S_summ, M_summ, names, y_coords, batch_size, nb_steps, window_shape,
                                           nb_max_augment, scores_path):
            # the previous batch's kernel has consumed ddesc once the stream reaches this copy (same stream, in order);
            # hdesc is reused only after the copy that read it has finished
            torch.cuda.current_stream(dev).synchronize()
            hdesc.copy_(torch.from_numpy(desc))
            ddesc.copy_(hdesc, non_blocking=True)
            ops.crop_batch(iptr, mptr, wid, ddesc, n, xb, yb)
            yield xb, yb

    # ------------------------------------------------------------------ predict / evaluate
    def predict(self, dataset_paths, model_path, window_shape=(512, 512), print_scores=False,
                save=False, augmentation=False, threshold=0.5):
        """unet_2d_summary.py:532-625.  Returns (Mp: list of uint8 masks [hs,ws], names)."""
        import torch
        logger = logging.getLogger(funcname())
        model = model_path if isinstance(model_path, UNetModel) else \
            load_model_with_new_input_shape(model_path, window_shape, compile=False, trainable=False)
        assert tuple(window_shape) == (512, 512), 'TODO: implement variable window sizes.'
        Mp, names = [], []
        mean_prec, mean_reca, mean_comb = 0., 0., 0.
        # Two-deep software pipeline over the datasets: while the GPU runs image i, the host loads / standardises image
        # i+1 and copies it from pinned memory STRAIGHT INTO the engine's static input buffer of the other slot (upload
        # stream); the mask of image i leaves through a pinned buffer on a download stream.  The compute stream carries
        # nothing but the captured step (no staging copies between two steps).  Results are identical to the serial loop
        # of the reference (:578-595).
        dev = model.engine.dev
        # the streams and the pinned staging buffers live on the engine and are reused by later predict() calls: pinned
        # allocations are slow (cudaHostAlloc maps the pages for every visible GPU - ~75 ms per call with 2 ranks on an
        # 8-GPU box, which was the whole difference between the device-timed and the end-to-end number at N >= 2)
        cache = model.engine.__dict__.setdefault('_predict_staging', {})
        if 'up' not in cache:
            cache['up'] = torch.cuda.Stream(device=dev)
            cache['down'] = torch.cuda.Stream(device=dev)
            cache['slots'] = [{}, {}]
            cache['score'] = torch.cuda.Stream(device=dev)
        up_stream, down_stream, slots, score_stream = cache['up'], cache['down'], cache['slots'], cache['score']

        def stage(i):
            dsp = dataset_paths[i]
            summ = np.ascontiguousarray(np.asarray(self.series_summary_func(dsp), dtype=np.float32))
            sl = slots[i % 2]
            # an image larger than the window is predicted from overlapping tiles (engine.predict_tiled), outside the
            # pipeline: its own compute dwarfs the staging this pipeline hides
            sl['large'] = summ.shape[0] > window_shape[0] or summ.shape[1] > window_shape[1]
            if sl['large']:
                sl['summ'] = summ
                return
            cfg = (summ.shape, bool(augmentation), float(threshold))
            if sl.get('cfg') != cfg:
                bufs = model.engine.tta_buffers(summ.shape, window=window_shape[0], augmentation=augmentation,
                                                threshold=threshold, slot=i % 2)
                sl.update(cfg=cfg, hin=torch.empty(summ.shape, dtype=torch.float32).pin_memory(),
                          din=bufs['summ'], dmask=bufs['mask'],
                          hout=torch.empty(summ.shape, dtype=torch.uint8).pin_memory(),
                          ready=torch.cuda.Event(), computed=torch.cuda.Event(), done=torch.cuda.Event())
                # buffers that were just created belong to the compute stream (their zero fill is queued there, and the
                # allocator may have handed out memory that queued work still reads): the first upload waits for it
                fresh = torch.cuda.Event()
                fresh.record(torch.cuda.current_stream(dev))
                up_stream.wait_event(fresh)
            # plain memcpy into the pinned buffer: torch's CPU copy_ goes through the OpenMP pool, and a pool as wide as the
            # machine next to another busy process (a second rank) turned this 1 MB copy into milliseconds
            np.copyto(sl['hin'].numpy(), summ)
            # the previous user of this slot's device buffers (image i - 2) was collected before this call
            with torch.cuda.stream(up_stream):
                sl['din'].copy_(sl['hin'], non_blocking=True)
                sl['ready'].record(up_stream)
            sl['summ'] = summ

        scores = [0., 0., 0.]

        def finalize(i):
            """image i has been enqueued earlier: wait for its mask (pinned buffer) and do the host-side bookkeeping"""
            dsp = dataset_paths[i]
            name = self.dataset_name_func(dsp)
            sl = slots[i % 2]
            if sl['large']:
                mp = sl.pop('mp')
            else:
                sl['done'].synchronize()
                mp = sl['hout'].numpy().copy()
            Mp.append(mp)
            names.append(name)
            m = None
            if print_scores:
                # scored on a stream of its own: waiting for the scores must not wait for image i, already queued
                m = self.mask_summary_func(dsp)
                with torch.cuda.stream(score_stream):
                    truth = torch.from_numpy(np.ascontiguousarray(np.asarray(m) != 0, dtype=np.uint8)).to(dev)
                    p, r, incl, excl, comb = nf_mask_metrics_device([(truth, torch.from_numpy(mp).to(dev))])[0]
                logger.info('%s: prec=%.3lf, reca=%.3lf, incl=%.3lf, excl=%.3lf, comb=%.3lf' % (name, p, r, incl, excl, comb))
                for k, v in enumerate((p, r, comb)):
                    scores[k] += v / len(dataset_paths)
            if save:                                   # outlined figure (:610-619): truth in blue when the dataset has masks
                from PIL import Image
                ds = open_dataset(dsp, keys=('masks/raw',)) if isinstance(dsp, str) and path.exists(dsp) else {}
                if 'masks/raw' in ds:
                    m = self.mask_summary_func(dsp) if m is None else m
                    outlined = _un.mask_outlines(sl['summ'], [m, mp.round()], ['blue', 'red'])
                else:
                    outlined = _un.mask_outlines(sl['summ'], [mp.round()], ['red'])
                save_path = '%s/%s_mp.png' % (self.cpdir, name)
                Image.fromarray(outlined).save(save_path)
                logger.info('Saved %s' % save_path)

        if len(dataset_paths):
            stage(0)
        for i, dsp in enumerate(dataset_paths):
            sl = slots[i % 2]
            if sl['large']:
                # the mask leaves before the next image runs: a later image of the same shape reuses its buffers
                mask, _ = model.engine.predict_tiled(torch.from_numpy(sl['summ']).to(dev), augmentation=augmentation,
                                                     threshold=threshold)
                sl['mp'] = mask.cpu().numpy()
            else:
                main = torch.cuda.current_stream(dev)
                main.wait_event(sl['ready'])
                model.engine.predict_tta(sl['din'], window=window_shape[0], augmentation=augmentation, threshold=threshold,
                                         slot=i % 2)
                sl['computed'].record(main)
                with torch.cuda.stream(down_stream):       # this slot's mask buffer is not touched again before finalize(i)
                    down_stream.wait_event(sl['computed'])
                    sl['hout'].copy_(sl['dmask'], non_blocking=True)
                    sl['done'].record(down_stream)
            # image i is now queued on the GPU; meanwhile collect image i-1 (frees its slot) and stage image i+1 into it
            if i >= 1:
                finalize(i - 1)
            if i + 1 < len(dataset_paths):
                stage(i + 1)
        if len(dataset_paths):
            finalize(len(dataset_paths) - 1)
        mean_prec, mean_reca, mean_comb = scores
        if print_scores:
            logger.info('Mean prec=%.3lf, reca=%.3lf, comb=%.3lf' % (mean_prec, mean_reca, mean_comb))
            self.last_scores = dict(prec=mean_prec, reca=mean_reca, comb=mean_comb)
        return Mp, names

    def evaluate(self, dataset_paths, model_path, window_shape=(512, 512), threshold=0.5):
        """The reference CLI's evaluation() (examples/neurons/unet2ds_nf.py:47-64): predict with and
        without test-time augmentation, printing scores.  Returns {augmentation flag: scores}."""
        out = {}
        for aug in (True, False):
            self.predict(dataset_paths, model_path, window_shape, print_scores=True, save=False,
                         augmentation=aug, threshold=threshold)
            out[aug] = dict(self.last_scores)
        return out
