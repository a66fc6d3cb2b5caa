"""Executor of the UNet2DS graph on one B200: sequences libdcb200 kernels for inference
(BatchNorm folded into the conv epilogues, optional 8x TTA) and for one Keras-style
``train_on_batch`` (batch-statistic BatchNorm, dropout, loss, backward, Adam), each
captured once into a CUDA graph and replayed.

Reference behaviour: deepcalcium/models/neurons/unet_2d_summary.py:123-224 (graph),
:429 (fit_generator -> train_on_batch), :585-595 (predict with TTA).
torch only owns memory / streams / graphs here; there is no torch arithmetic on the path.
"""
from collections import OrderedDict

import os

import numpy as np
import torch

from .. import _native as nat
from . import ops
from .graph import (GraphSpec, BN_EPS, BN_MOMENTUM_CONV, BN_MOMENTUM_UP, flat_layout, he_normal_weights, pack, pack_flat,
                    plan_tiles, tile_halo, tile_limits, unpack, unpack_flat)

_PRECISIONS = {'bf16': torch.bfloat16, 'fp16': torch.float16, 'f16': torch.float16, 'fp32': torch.float32, 'f32': torch.float32}


def _on_engine_device(fn):
    """run a public engine method with the engine's device current: the C-ABI wrappers enqueue on the CURRENT device's
    stream, which must be the device that owns the engine's buffers"""
    import functools

    @functools.wraps(fn)
    def wrapper(self, *a, **k):
        with torch.cuda.device(self.dev):
            return fn(self, *a, **k)
    return wrapper


class UNetEngine(object):
    def __init__(self, spec=None, precision='bf16', device=None, use_graphs=True):
        nat.require_cuda()
        self.spec = spec or GraphSpec()
        self.dtype = _PRECISIONS[precision]
        # 'bf16' / 'fp16': tcgen05 kernels (fp16 = inference only: same MMA rate, 10 mantissa bits instead of 7, meets the
        # north star's 1e-2 logit tolerance where bf16 storage cannot); 'fp32': CUDA-core check mode
        self.precision = {torch.bfloat16: 'bf16', torch.float16: 'fp16', torch.float32: 'fp32'}[self.dtype]
        self.tc = self.dtype != torch.float32
        # what the kernels run: the 16-bit precisions pad every channel width (graph.padded_width), the fp32 check mode
        # runs the spec as it is.  Weights and optimiser state cross the engine's boundary in the layout of self.spec.
        self.dspec = self.spec.device_spec(self.precision)
        self.head_c = self.dspec.by_name['head'].cin
        self.dev = torch.device(device if device is not None else 'cuda:%d' % torch.cuda.current_device())
        self.use_graphs = use_graphs
        self._build_param_storage()
        self._build_derived()
        self._inputs = self._wire()
        self._weights_dirty = True
        self._sessions = {}
        self._prep_tables = {}
        # every encoder block's 2x2 max-pool is folded into the producing conv's epilogue (strip kernel: Cout <= 64 on wide
        # rows; generic kernel: both orientations); no standalone pooling launch in inference
        self._pool_fused = ('enc0b', 'enc1b', 'enc2b', 'enc3b')
        self.iteration = 0
        self.launches = 0
        self.comm = None          # engine.dist.Comm for data-parallel training (None = single GPU)
        self.overlap_wgrad = True  # weight-gradient launches on a side stream (see _train_step_enqueue)
        self.rank1_head_grad = True   # the softmax head's input gradient stays factored (see _train_step_enqueue)
        self.head_wd = torch.zeros(self.head_c, dtype=torch.float32, device=self.dev)
        self.pdl = os.environ.get('DCB_PDL', '1') != '0'   # programmatic dependent launch in the inference forward
        # ... along the main chain of the training step it LOSES (2.81 -> 3.14 ms, scripts/train_time.py): the early-resident
        # CTAs of the next main-chain kernel take the SM slots in which the weight-gradient side stream overlapped
        self.pdl_train = os.environ.get('DCB_PDL_TRAIN', '0') != '0'
        self._side = None
        self.halo = tile_halo(self.spec)
        # predict_tiled runs its tiles in groups of at most this many batch pixels, tiles of at most max_tile pixels a side
        # (8 transforms of one 2048^2 tile up to nb_filters_base 32; the same activation bytes for wider networks)
        self.tile_batch_pixels, self.max_tile = tile_limits(self.dspec, self.dtype.itemsize)
        self.set_weights_dict(he_normal_weights(self.spec, seed=0))

    # ------------------------------------------------------------------ parameter storage
    def _build_param_storage(self):
        self._slots, off_t, off_n = flat_layout(self.dspec)        # key -> (trainable?, offset, device shape)
        f32 = dict(dtype=torch.float32, device=self.dev)
        self.params = torch.zeros(off_t, **f32)
        self.grads = torch.zeros(off_t, **f32)
        self.adam_m = torch.zeros(off_t, **f32)
        self.adam_v = torch.zeros(off_t, **f32)
        self.nontrain = torch.zeros(max(off_n, 4), **f32)
        self.P, self.G = OrderedDict(), OrderedDict()
        for key, (tr, off, shp) in self._slots.items():
            n = int(np.prod(shp))
            base = self.params if tr else self.nontrain
            self.P[key] = base[off:off + n].view(*shp)
            if tr:
                self.G[key] = self.grads[off:off + n].view(*shp)
        # device-resident step state {iteration, dropout seed} and lr_t (see dcb_step_advance)
        self.step_state = torch.zeros(2, dtype=torch.int64, device=self.dev)
        self.lr_t = torch.zeros(1, **f32)

    def _build_derived(self):
        f32 = dict(dtype=torch.float32, device=self.dev)
        T = dict(dtype=self.dtype, device=self.dev)
        self.w_fwd, self.w_dgrad = {}, {}
        self.inf_scale, self.inf_shift = {}, {}
        self.bn = {}
        n_dbl = 0
        for blk in self.dspec.blocks:
            if blk.kind == 'head':
                continue
            nk = int(np.prod(blk.kernel_shape()))
            k = self.P[blk.name + '/kernel']
            if blk.kind == 'conv':
                if blk.cin == 1 and self.tc:
                    self.w_fwd[blk.name] = k                     # c1 kernel reads the fp32 master
                    self.w_dgrad[blk.name] = None
                elif self.dtype == torch.float32:
                    self.w_fwd[blk.name] = k                     # fp32 layout == Keras HWIO
                    self.w_dgrad[blk.name] = torch.empty(nk, **T) if blk.cin > 1 else None
                else:
                    self.w_fwd[blk.name] = torch.empty(nk, **T)
                    self.w_dgrad[blk.name] = torch.empty(nk, **T)
            else:
                if self.dtype == torch.float32:
                    self.w_fwd[blk.name] = torch.empty(nk, **T)
                    self.w_dgrad[blk.name] = k                   # fp32 dgrad layout == Keras (2,2,Cout,Cin)
                else:
                    self.w_fwd[blk.name] = torch.empty(nk, **T)
                    self.w_dgrad[blk.name] = torch.empty(nk, **T)
            self.inf_scale[blk.name] = torch.empty(blk.cout, **f32)
            self.inf_shift[blk.name] = torch.empty(blk.cout, **f32)
            self.bn[blk.name] = dict(scale=torch.empty(blk.cout, **f32), shift=torch.empty(blk.cout, **f32),
                                     mean=torch.empty(blk.cout, **f32), rstd=torch.empty(blk.cout, **f32),
                                     off_f=n_dbl, off_b=n_dbl + 2 * blk.cout)
            n_dbl += 4 * blk.cout
        self._off_head_sums = n_dbl
        self._off_head_dwb = n_dbl + 8
        n_dbl += 8 + 2 * self.head_c + 2
        self.dbl = torch.zeros(n_dbl, dtype=torch.float64, device=self.dev)
        # single-launch BatchNorm kernels (dcb_bn_train_fwd / _bwd): 4 barrier words per (layer, direction), zeroed at the
        # start of every step, and one shared workspace for the fixed-point per-channel totals (zeroed once; the kernels
        # leave it zeroed)
        self.bn_sync = torch.zeros(8 * len(self.dspec.blocks), dtype=torch.int32, device=self.dev)
        self.bn_ws = torch.zeros(ops.bn_train_workspace_bytes(max(b.cout for b in self.dspec.blocks)), dtype=torch.uint8,
                                 device=self.dev)
        self.peers = None         # dcb_peer_exchange description for in-kernel SyncBN (engine.dist.attach_peers)
        self.metrics = torch.zeros(8, **f32)

    def _wire(self):
        inp = OrderedDict()
        inp['enc0a'] = ('x', None); inp['enc0b'] = ('enc0a', None)
        for l in (1, 2, 3):
            inp['enc%da' % l] = ('pool%d' % (l - 1), None); inp['enc%db' % l] = ('enc%da' % l, None)
        inp['bota'] = ('pool3', None); inp['botb'] = ('bota', None)
        prev = 'botb'
        self._ups = OrderedDict()          # 'upsampling' mode: up<l> = nearest 2x of prev (+dropout), not a weight layer
        for l in (3, 2, 1, 0):
            if self.spec.up_mode == 'transpose':
                inp['up%d' % l] = (prev, None)
            else:
                self._ups['up%d' % l] = prev
            inp['dec%da' % l] = ('up%d' % l, 'enc%db' % l)
            inp['dec%db' % l] = ('dec%da' % l, None)
            prev = 'dec%db' % l
        inp['head'] = ('dec0b', None)
        return inp

    # ------------------------------------------------------------------ weights in / out (Keras layouts)
    def set_weights_dict(self, w):
        shapes = self.spec.weight_shapes()
        real = OrderedDict()
        for key, shp in shapes.items():
            real[key] = np.asarray(w[key], dtype=np.float32)
            if tuple(real[key].shape) != tuple(shp):
                raise ValueError('weight %s: expected shape %s, got %s' % (key, shp, real[key].shape))
        for key, a in pack(self.spec, self.dspec, real).items():
            self.P[key].copy_(torch.from_numpy(np.ascontiguousarray(a)))
        self._weights_dirty = True

    def get_weights_dict(self):
        torch.cuda.synchronize(self.dev)
        return unpack(self.spec, self.dspec, OrderedDict((key, self.P[key].detach().cpu().numpy().copy()) for key in self._slots))

    def get_optimizer_state(self):
        """Adam's m and v over the trainable parameters in flat_layout(self.spec) - the layout of an unpadded engine,
        so the state moves between precisions - and the step state {iteration, dropout seed}."""
        torch.cuda.synchronize(self.dev)
        m, v = (unpack_flat(self.spec, self.dspec, t.cpu().numpy()) for t in (self.adam_m, self.adam_v))
        return OrderedDict(adam_m=m, adam_v=v, step_state=self.step_state.cpu().numpy())

    def set_optimizer_state(self, adam_m, adam_v, step_state):
        """inverse of get_optimizer_state"""
        self.adam_m.copy_(torch.from_numpy(pack_flat(self.spec, self.dspec, adam_m)))
        self.adam_v.copy_(torch.from_numpy(pack_flat(self.spec, self.dspec, adam_v)))
        self.step_state.copy_(torch.from_numpy(np.asarray(step_state, dtype=np.int64)))
        self.iteration = int(step_state[0])

    def reset_optimizer(self):
        self.adam_m.zero_(); self.adam_v.zero_()
        self.step_state.zero_()
        self.iteration = 0

    def _prep_table(self, for_training):
        """device table for dcb_prep_weights_batch (built once per mode; the buffers are static)."""
        tab = self._prep_tables.get(for_training)
        if tab is None:
            rows = []
            for blk in self.dspec.blocks:
                if blk.kind == 'head':
                    continue
                n = blk.name
                k = self.P[n + '/kernel']
                if blk.kind == 'conv':
                    wf = self.w_fwd[n] if self.w_fwd[n] is not k else None
                    wd = self.w_dgrad[n] if for_training else None
                else:
                    wf = self.w_fwd[n]
                    wd = self.w_dgrad[n] if (for_training and self.w_dgrad[n] is not k) else None
                if wf is None and wd is None:
                    continue
                cin, cout = (k.shape[2], k.shape[3]) if blk.kind == 'conv' else (k.shape[3], k.shape[2])
                rows.append([k.data_ptr(), wf.data_ptr() if wf is not None else 0, wd.data_ptr() if wd is not None else 0,
                             cin | (cout << 32), 0 if blk.kind == 'conv' else 1])
            tab = (torch.tensor(rows, dtype=torch.int64, device=self.dev), len(rows)) if rows else (None, 0)
            self._prep_tables[for_training] = tab
        return tab

    def _prepare_weights(self, for_training):
        """fold BN for inference and (re)build the kernel-layout weight copies."""
        tab, count = self._prep_table(for_training)
        if count:
            ops.prep_weights_batch(tab, count, self.dtype)
        if for_training:
            return
        for blk in self.dspec.blocks:
            if blk.kind == 'head':
                continue
            n = blk.name
            if not for_training:
                ops.bn_fold(self.P[n + '/gamma'], self.P[n + '/beta'], self.P[n + '/moving_mean'],
                            self.P[n + '/moving_var'], self.P[n + '/bias'], self.inf_scale[n], self.inf_shift[n], BN_EPS)

    # ------------------------------------------------------------------ activation buffers
    def _session(self, NB, H, W, training):
        key = (NB, H, W, training)
        s = self._sessions.get(key)
        if s is not None:
            return s
        if H % 16 or W % 16:
            raise ValueError('window %dx%d must be a multiple of 16 (four 2x2 poolings)' % (H, W))
        T = dict(dtype=self.dtype, device=self.dev)
        s = dict(NB=NB, H=H, W=W, training=training, act={}, raw={}, dx={}, graph=None, tta_graphs={})
        s['x'] = torch.zeros(NB, H, W, dtype=torch.float32, device=self.dev)
        if self.dtype == torch.float32:
            s['act']['x'] = s['x'].view(NB, H, W, 1)
        for blk in self.dspec.blocks:
            if blk.kind == 'head':
                continue
            h, w = H >> blk.level, W >> blk.level
            s['act'][blk.name] = torch.empty(NB, h, w, blk.cout, **T)
            if training:
                s['raw'][blk.name] = torch.empty(NB, h, w, blk.cout, **T)
                if blk.name != 'enc0a':
                    # gradient tensors are fp32 in both precisions (see dcb_conv3x3_dgrad)
                    if blk.kind == 'conv':
                        s['dx'][blk.name] = torch.empty(NB, h, w, blk.cin, dtype=torch.float32, device=self.dev)
                    else:
                        s['dx'][blk.name] = torch.empty(NB, h // 2, w // 2, blk.cin, dtype=torch.float32, device=self.dev)
        for un, prev in self._ups.items():
            l = int(un[2:])
            c = self.dspec.by_name[prev].cout
            s['act'][un] = torch.empty(NB, H >> l, W >> l, c, **T)
            if training:
                s['dx'][un] = torch.empty(NB, H >> (l + 1), W >> (l + 1), c, dtype=torch.float32, device=self.dev)
        for l in range(4):
            c = self.dspec.by_name['enc%db' % l].cout
            s['act']['pool%d' % l] = torch.empty(NB, H >> (l + 1), W >> (l + 1), c, **T)
            if training:
                s['dx']['skip%d' % l] = torch.empty(NB, H >> l, W >> l, c, dtype=torch.float32, device=self.dev)
        s['logit'] = torch.empty(NB, H, W, dtype=torch.float32, device=self.dev)
        s['prob'] = torch.empty(NB, H, W, dtype=torch.float32, device=self.dev)
        if training:
            s['y'] = torch.zeros(NB, H, W, dtype=torch.uint8, device=self.dev)
            s['dhead'] = torch.empty(NB, H, W, self.head_c, dtype=torch.float32, device=self.dev)
            s['gpix'] = torch.empty(NB, H, W, dtype=torch.float32, device=self.dev)     # rank-1 head gradient: per-pixel factor
            need = 0
            for blk in self.dspec.blocks:
                h, w = H >> blk.level, W >> blk.level
                if blk.kind == 'conv':
                    if blk.cin == 1 and self.tc:
                        need = max(need, ops.conv3x3_c1_wgrad_workspace_bytes(blk.cout))
                    else:
                        need = max(need, ops.conv3x3_wgrad_workspace_bytes(self.dtype, NB, h, w, blk.cin, blk.cout))
                elif blk.kind == 'up':
                    need = max(need, ops.convT2x2_wgrad_workspace_bytes(self.dtype, NB, h // 2, w // 2, blk.cin, blk.cout))
            # one workspace per session: a captured training graph keeps the pointer it was recorded with
            s['wgrad_ws'] = torch.empty(max(need, 16), dtype=torch.uint8, device=self.dev)
        self._sessions[key] = s
        return s

    # ------------------------------------------------------------------ inference
    def _forward_inference(self, s, prob_out=None):
        """enqueue the forward pass reading s['x'] (fp32 [NB,H,W]); writes s['logit'] and s['prob'] (or ``prob_out``: any
        [NB,H,W] fp32 device buffer, e.g. a slice of another rank's peer-mapped result buffer).
        The max-pool after each encoder block and the softmax head are folded into the producing conv's
        epilogue (dcb_conv3x3_fwd_fused) - the library falls back to the separate kernels where the fused
        epilogue does not apply."""
        # programmatic dependent launch: every kernel of the inference forward reads only static data (weights, folded BN
        # coefficients) before its dependency wait, so consecutive layers overlap prologue and tail
        with nat.policy(pdl=1 if self.pdl else 0):
            self._forward_inference_enqueue(s, prob_out)

    def _forward_inference_enqueue(self, s, prob_out):
        act = s['act']
        for blk in self.dspec.blocks:
            n = blk.name
            if blk.kind == 'head':
                continue                                  # fused into dec0b below
            a, b = self._inputs[n]
            sc, sh = self.inf_scale[n], self.inf_shift[n]
            if a in self._ups:
                ops.upsample2x(act[self._ups[a]], act[a])
            if blk.kind == 'conv':
                if blk.cin == 1 and self.tc:
                    ops.conv3x3_c1_fwd(s['x'], self.w_fwd[n], act[n], sc, sh, True)
                elif n == 'dec0b':
                    ops.conv3x3_fwd_fused(act[a], None, self.w_fwd[n], act[n], sc, sh, True,
                                          head_kernel=self.P['head/kernel'], head_bias=self.P['head/bias'],
                                          logit=s['logit'], prob=prob_out if prob_out is not None else s['prob'], need_y=False)
                elif n in self._pool_fused and self.tc:
                    # the 2x2 max-pool rides in the conv epilogue where the layer runs on the (folded) strip kernel
                    ops.conv3x3_fwd_fused(act[a], None, self.w_fwd[n], act[n], sc, sh, True, pool_out=act['pool%d' % blk.level])
                else:
                    ops.conv3x3_fwd(act[a], act[b] if b else None, self.w_fwd[n], act[n], sc, sh, True)
                    if n in ('enc0b', 'enc1b', 'enc2b', 'enc3b'):
                        ops.maxpool2x2(act[n], act['pool%d' % blk.level])
            else:
                ops.convT2x2_fwd(act[a], self.w_fwd[n], act[n], sc, sh, True)

    def _ensure_inference_ready(self):
        if self._weights_dirty:
            self._prepare_weights(for_training=False)
            self._weights_dirty = False

    def _run_graphed(self, holder, key, fn):
        """run fn() through a CUDA graph cached in holder[key] (first call: eager warm-up then capture)."""
        # Every call executes fn's work exactly once (a training step mutates state):
        # call 1 runs eagerly (also builds the TMA descriptor caches), call 2 captures and replays,
        # later calls replay.
        # self.launches counts the library's kernel launches including those replayed from graphs.
        c0 = nat.launch_count()
        if not self.use_graphs:
            fn()
            self.launches += nat.launch_count() - c0
            return
        g = holder.get(key)
        if g is None:
            fn()
            self.launches += nat.launch_count() - c0
            holder[key] = 'warm'
            return
        if isinstance(g, str):
            torch.cuda.synchronize(self.dev)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                fn()
            g.dcb_launches = nat.launch_count() - c0
            holder[key] = g
        g.replay()
        self.launches += g.dcb_launches

    @_on_engine_device
    def infer(self, x_dev):
        """x_dev: fp32 CUDA tensor [NB,H,W].  Returns (prob, logit) fp32 [NB,H,W] (views of static buffers)."""
        NB, H, W = x_dev.shape
        s = self._session(NB, H, W, False)
        self._ensure_inference_ready()
        s['x'].copy_(x_dev)
        self._run_graphed(s, 'graph', lambda: self._forward_inference(s))
        return s['prob'], s['logit']

    def _tta_state(self, hs, ws, window, augmentation, threshold, transforms, slot):
        n_aug = 8 if augmentation else 1
        first, count = transforms if transforms is not None else (0, n_aug)
        s = self._session(count, window, window, False)
        key = (hs, ws, n_aug, first, count, float(threshold), transforms is None, slot)
        st = s['tta_graphs'].get(('bufs',) + key)
        if st is None:
            st = dict(summ=torch.zeros(hs, ws, dtype=torch.float32, device=self.dev),
                      mask=torch.zeros(hs, ws, dtype=torch.uint8, device=self.dev),
                      act=torch.zeros(hs, ws, dtype=torch.float64, device=self.dev))
            s['tta_graphs'][('bufs',) + key] = st
        return s, key, st, n_aug, first, count

    @_on_engine_device
    def tta_buffers(self, shape, window=512, augmentation=True, threshold=0.5, slot=0):
        """the static input / output buffers of predict_tta for (shape, slot): a caller that pipelines images copies the
        next summary image straight into ``summ`` of the OTHER slot (and reads ``mask`` of a finished one) while a step
        runs; predict_tta(buffers['summ'], ..., slot=slot) then skips its device-to-device input copy."""
        return self._tta_state(shape[0], shape[1], window, augmentation, threshold, None, slot)[2]

    @_on_engine_device
    def predict_tta(self, summ_dev, window=512, augmentation=True, threshold=0.5, transforms=None, slot=0):
        """unet_2d_summary.py:578-595 for one summary image already on the device (fp32 [hs,ws]).
        Returns (mask uint8 [hs,ws], act float64 [hs,ws]) as device tensors (static buffers).
        ``transforms`` = (first, count) restricts the batch to a slice of the 8 transforms and skips
        the combine (multi-GPU sharding, returns the raw probabilities [count,S,S]).
        ``slot`` selects one of several independent sets of static input / output buffers (and captured graphs) that
        share the activation buffers: see tta_buffers."""
        hs, ws = summ_dev.shape
        s, key, st, n_aug, first, count = self._tta_state(hs, ws, window, augmentation, threshold, transforms, slot)
        self._ensure_inference_ready()
        if summ_dev.data_ptr() != st['summ'].data_ptr():
            st['summ'].copy_(summ_dev)

        def run():
            with nat.policy(pdl=1 if self.pdl else 0):
                ops.tta_make_batch(st['summ'], window, first, count, s['x'])
                self._forward_inference(s)
                if transforms is None:
                    ops.tta_combine(s['prob'], window, hs, ws, threshold, n_aug, st['act'], st['mask'])

        self._run_graphed(s['tta_graphs'], key, run)
        if transforms is not None:
            return s['prob']
        return st['mask'], st['act']

    def _batch_prefix(self, s, nb):
        """session s restricted to its first nb images (views of its buffers): the last, smaller group of a tile plan"""
        if nb == s['NB']:
            return s
        v = s.setdefault('prefixes', {}).get(nb)
        if v is None:
            v = dict(NB=nb, H=s['H'], W=s['W'], training=False, x=s['x'][:nb], logit=s['logit'][:nb], prob=s['prob'][:nb],
                     act={k: a[:nb] for k, a in s['act'].items()})
            s['prefixes'][nb] = v
        return v

    @_on_engine_device
    def predict_tiled(self, summ_dev, augmentation=True, threshold=0.5, tile=None):
        """predict_tta for a summary image of any size (fp32 [hs,ws] on the device): the reference's TTA computed on the
        canvas (the image reflect-padded at the bottom and right to C_h x C_w, C_d = max(T, roundup16(size_d))) and cropped
        to hs x ws.  The canvas runs as square T x T tiles (graph.plan_tiles; ``tile=None`` picks T) that overlap by the
        network's receptive reach, so every pixel gets exactly the whole-canvas prediction from the one tile that owns
        it.  Tiles go through the 8-transform batch in groups of at most tile_batch_pixels batch pixels; one CUDA graph
        holds every group.  Returns (mask uint8 [hs,ws], act float64 [hs,ws]) as device tensors (static buffers)."""
        hs, ws = summ_dev.shape
        plan = plan_tiles((hs, ws), self.halo, tile, self.max_tile)
        T, n_aug = plan.tile, (8 if augmentation else 1)
        per_group = min(plan.n_tiles, max(1, self.tile_batch_pixels // (n_aug * T * T)))
        s = self._session(per_group * n_aug, T, T, False)
        key = ('tiled', n_aug, float(threshold), plan.key())
        st = s['tta_graphs'].get(('bufs',) + key)
        if st is None:
            i32 = dict(dtype=torch.int32, device=self.dev)
            st = dict(summ=torch.zeros(hs, ws, dtype=torch.float32, device=self.dev),
                      mask=torch.zeros(hs, ws, dtype=torch.uint8, device=self.dev),
                      act=torch.zeros(hs, ws, dtype=torch.float64, device=self.dev),
                      oy=torch.tensor(plan.origins[0], **i32), ox=torch.tensor(plan.origins[1], **i32),
                      cy=torch.tensor(plan.cuts[0], **i32), cx=torch.tensor(plan.cuts[1], **i32))
            s['tta_graphs'][('bufs',) + key] = st
        self._ensure_inference_ready()
        st['summ'].copy_(summ_dev)

        def run():
            with nat.policy(pdl=1 if self.pdl else 0):
                for t0 in range(0, plan.n_tiles, per_group):
                    nt = min(per_group, plan.n_tiles - t0)
                    g = self._batch_prefix(s, nt * n_aug)
                    ops.tile_make_batch(st['summ'], T, st['oy'], st['ox'], t0, nt, 0, n_aug, g['x'])
                    self._forward_inference(g)
                    ops.tile_combine(g['prob'], T, st['oy'], st['ox'], st['cy'], st['cx'], t0, nt, threshold, n_aug,
                                     st['act'], st['mask'])

        self._run_graphed(s['tta_graphs'], key + (per_group,), run)
        return st['mask'], st['act']

    # ------------------------------------------------------------------ training
    def _side_stream(self):
        if self._side is None:
            self._side = torch.cuda.Stream(device=self.dev)
        return self._side

    def _dropout_p(self, name, enabled):
        return float(self.spec.dropout_after().get(name, 0.)) if enabled else 0.

    def _allreduce(self, t):
        if self.comm is not None and self.comm.world > 1:
            self.comm.allreduce_sum(t)

    def _train_step_enqueue(self, s, loss_id, lr, dropout, beta1, beta2, eps):
        spec, act, raw, dxb = self.dspec, s['act'], s['raw'], s['dx']
        world = self.comm.world if self.comm is not None else 1
        # ranks draw different dropout masks for their own crops
        seed_base = (self.comm.rank if self.comm is not None else 0) * 0x9E3779B1
        seed_dev = self.step_state[1:2]
        ops.step_advance(self.step_state, lr, beta1, beta2, self.lr_t)
        self.dbl.zero_()
        # fused single-launch BatchNorm unless the policy says otherwise; a data-parallel run needs the peer-mapped
        # exchange buffers for it (otherwise: separate passes with NCCL all-reduces of the sums in between)
        fused_bn = bool(nat.get_policy('fused_bn')) and (world == 1 or self.peers is not None)
        if fused_bn:
            self.bn_sync.zero_()
        epi_stats = fused_bn and nat.get_policy('fused_bn') >= 2 and self.dtype == torch.bfloat16
        # the 16-bit kernel-layout copies of the updated weights are rebuilt on the side stream while the first layer
        # (which reads the fp32 master weights) and its BatchNorm run; the first tensor-core conv waits for them
        main = torch.cuda.current_stream(self.dev)
        side = self._side_stream() if self.overlap_wgrad else None
        prep_done = None
        if side is not None and self.tc:
            ev = torch.cuda.Event()
            ev.record(main)
            side.wait_event(ev)
            with torch.cuda.stream(side):
                self._prepare_weights(for_training=True)
                prep_done = torch.cuda.Event()
                prep_done.record(side)
        else:
            self._prepare_weights(for_training=True)
        layer_id = {blk.name: i for i, blk in enumerate(spec.blocks)}
        for i, un in enumerate(self._ups):
            layer_id[un] = len(spec.blocks) + i
        # ---------------- forward (batch-statistic BN)
        for blk in spec.blocks:
            n = blk.name
            if blk.kind == 'head':
                continue
            a, b = self._inputs[n]
            bias = self.P[n + '/bias']
            if a in self._ups:
                ops.upsample2x(act[self._ups[a]], act[a], self._dropout_p(a, dropout), seed_base, seed_dev, layer_id[a])
            st = self.bn[n]
            # batch statistics taken by the conv epilogue (fused_bn = 2, bf16): the BatchNorm launch that follows is a single
            # pass without grid barriers.  have_sums is decided by the library per shape (False: full single-launch kernel).
            # (the forward slot of the fp64 scratch, zeroed at the start of the step, read as 2^-20 fixed-point int64)
            fsums = self.dbl[st['off_f']:st['off_f'] + 2 * blk.cout].view(torch.int64)
            have_sums = False
            if blk.kind == 'conv':
                if blk.cin == 1 and self.tc:
                    if epi_stats:
                        have_sums = ops.conv3x3_c1_fwd_stats(s['x'], self.w_fwd[n], raw[n], fsums, None, bias, False)
                    else:
                        ops.conv3x3_c1_fwd(s['x'], self.w_fwd[n], raw[n], None, bias, False)
                else:
                    if prep_done is not None:
                        main.wait_event(prep_done)
                        prep_done = None
                    if epi_stats:
                        have_sums = ops.conv3x3_fwd_stats(act[a], act[b] if b else None, self.w_fwd[n], raw[n], fsums, None, bias, False)
                    else:
                        ops.conv3x3_fwd(act[a], act[b] if b else None, self.w_fwd[n], raw[n], None, bias, False)
                mom = BN_MOMENTUM_CONV
            else:
                if prep_done is not None:
                    main.wait_event(prep_done)
                    prep_done = None
                if epi_stats:
                    have_sums = ops.convT2x2_fwd_stats(act[a], self.w_fwd[n], raw[n], fsums, None, bias, False)
                else:
                    ops.convT2x2_fwd(act[a], self.w_fwd[n], raw[n], None, bias, False)
                mom = BN_MOMENTUM_UP
            M = raw[n].numel() // blk.cout
            pooled = act['pool%d' % blk.level] if n in ('enc0b', 'enc1b', 'enc2b', 'enc3b') else None
            if have_sums:
                li = layer_id[n]
                ops.bn_train_fwd_sums(raw[n], fsums, self.P[n + '/gamma'], self.P[n + '/beta'], mom, self.P[n + '/moving_mean'],
                                      self.P[n + '/moving_var'], st['scale'], st['shift'], st['mean'], st['rstd'], act[n], True,
                                      self._dropout_p(n, dropout), seed_base, seed_dev, li, pool_out=pooled, M_total=M * world,
                                      eps=BN_EPS, peers=self.peers, slot=2 * li)
                continue
            if fused_bn:
                # statistics + normalise + ReLU + dropout (+ the 2x2 max-pool of the encoder blocks) in ONE launch; in
                # data-parallel runs the per-channel sums of all ranks are exchanged inside the kernel (SyncBN over NVLink)
                li = layer_id[n]
                ops.bn_train_fwd(raw[n], self.P[n + '/gamma'], self.P[n + '/beta'], mom, self.P[n + '/moving_mean'],
                                 self.P[n + '/moving_var'], st['scale'], st['shift'], st['mean'], st['rstd'], act[n], self.bn_ws,
                                 self.bn_sync[8 * li:8 * li + 4], True, self._dropout_p(n, dropout), seed_base, seed_dev, li,
                                 pool_out=pooled, M_total=M * world, eps=BN_EPS, peers=self.peers, slot=2 * li)
                continue
            sums = self.dbl[st['off_f']:st['off_f'] + 2 * blk.cout]
            ops.bn_stats(raw[n], sums)
            self._allreduce(sums)                       # SyncBN: statistics of the global batch
            ops.bn_finalize_apply(raw[n], sums, M * world, self.P[n + '/gamma'], self.P[n + '/beta'], mom,
                                  self.P[n + '/moving_mean'], self.P[n + '/moving_var'], st['scale'], st['shift'], st['mean'],
                                  st['rstd'], act[n], True, self._dropout_p(n, dropout), seed_base, seed_dev, layer_id[n], BN_EPS)
            if pooled is not None:
                ops.maxpool2x2(act[n], pooled)
        # ---------------- head + loss + its gradient
        hs = self.dbl[self._off_head_sums:self._off_head_sums + 8]
        hc = self.head_c
        hd = self.dbl[self._off_head_dwb:self._off_head_dwb + 2 * hc + 2]
        ops.head_loss_fwd(act['dec0b'], self.P['head/kernel'], self.P['head/bias'], s['y'], s['prob'], hs)
        if self.peers is not None:                      # loss / metric sums of the global batch: one-shot exchange over NVLink
            ops.peer_allreduce_f64(hs, self.peers, self.peers['n_slots'] - 1)
        else:
            self._allreduce(hs)
        # head kernel [1,1,C,2] and bias [2] are adjacent in the flat gradient buffer
        off_k = self._slots['head/kernel'][1]
        dw_out = self.grads[off_k:off_k + 2 * hc + 2]
        assert self._slots['head/bias'][1] == off_k + 2 * hc
        # dL/d(dec0b) = gpix[pixel] * wd[channel] is never materialised when the single-launch BatchNorm backward follows: the
        # head kernel writes the two factors, dec0b's BatchNorm backward rebuilds the product while it reads (134 MB less to
        # write and 2 x 67 MB less to read for a 32 x 128^2 batch)
        rank1 = fused_bn and self.rank1_head_grad and hc == 32
        if rank1:
            ops.head_loss_bwd_rank1(act['dec0b'], self.P['head/kernel'], s['y'], s['prob'], hs, loss_id, s['gpix'], self.head_wd,
                                    hd, dw_out, self.metrics, M_total=s['prob'].numel() * world)
        else:
            ops.head_loss_bwd(act['dec0b'], self.P['head/kernel'], s['y'], s['prob'], hs, loss_id, s['dhead'], hd, dw_out,
                              self.metrics, M_total=s['prob'].numel() * world)
        # ---------------- backward
        # Weight gradients are off the critical path: layer L's wgrad needs only d_raw(L) and the saved input, and nothing
        # before the optimizer reads its result, while the chain BN-bwd(L) -> dgrad(L) -> BN-bwd(L-1) ... is strictly
        # sequential.  The wgrad launches therefore go to a side stream (forked / joined with events, so the whole step
        # is still one CUDA graph) and overlap with the memory-bound BatchNorm / pooling kernels of the main chain.
        main = torch.cuda.current_stream(self.dev)
        side = self._side_stream() if self.overlap_wgrad else None

        def on_wgrad_stream(fn, *args):
            if side is None:
                return fn(*args)
            ev = torch.cuda.Event()
            ev.record(main)
            side.wait_event(ev)
            with torch.cuda.stream(side):
                fn(*args)

        grad_of = {'dec0b': ((s['gpix'], self.head_wd) if rank1 else s['dhead'], hc, 0)}
        skip_grad = {}
        for blk in reversed(spec.blocks):
            n = blk.name
            if blk.kind == 'head':
                continue
            a, b = self._inputs[n]
            dy, ldy, offy = grad_of[n]
            st = self.bn[n]
            sums = self.dbl[st['off_b']:st['off_b'] + 2 * blk.cout]
            p = self._dropout_p(n, dropout)
            draw = raw[n]      # in place: raw is dead after this point
            if fused_bn and isinstance(dy, tuple):      # rank-1 gradient of the softmax head (dec0b)
                li = layer_id[n]
                ops.bn_train_bwd_rank1(dy[0], dy[1], raw[n], st['scale'], st['shift'], st['mean'], st['rstd'], draw,
                                       self.G[n + '/gamma'], self.G[n + '/beta'], self.bn_ws, self.bn_sync[8 * li + 4:8 * li + 8], p,
                                       seed_base, seed_dev, li, M_total=(raw[n].numel() // blk.cout) * world, dgb_scale=1.0 / world,
                                       peers=self.peers, slot=2 * li + 1)
            elif fused_bn:
                li = layer_id[n]
                ops.bn_train_bwd(dy, ldy, offy, raw[n], st['scale'], st['shift'], st['mean'], st['rstd'], draw,
                                 self.G[n + '/gamma'], self.G[n + '/beta'], self.bn_ws, self.bn_sync[8 * li + 4:8 * li + 8], p,
                                 seed_base, seed_dev, li, M_total=(raw[n].numel() // blk.cout) * world, dgb_scale=1.0 / world,
                                 peers=self.peers, slot=2 * li + 1)
            else:
                ops.bn_bwd_reduce(dy, ldy, offy, raw[n], st['scale'], st['shift'], st['mean'], st['rstd'], sums, p, seed_base,
                                  seed_dev, layer_id[n])
                self._allreduce(sums)
                ops.bn_bwd_apply(dy, ldy, offy, raw[n], st['scale'], st['shift'], st['mean'], st['rstd'], sums, draw,
                                 self.G[n + '/gamma'], self.G[n + '/beta'], p, seed_base, seed_dev, layer_id[n],
                                 M_total=(raw[n].numel() // blk.cout) * world, dgb_scale=1.0 / world)
            if blk.kind == 'conv':
                if blk.cin == 1 and self.tc:
                    on_wgrad_stream(ops.conv3x3_c1_wgrad, s['x'], draw, self.G[n + '/kernel'], s['wgrad_ws'])
                else:
                    on_wgrad_stream(ops.conv3x3_wgrad, act[a], act[b] if b else None, draw, self.G[n + '/kernel'], s['wgrad_ws'])
                if n == 'enc0a':
                    continue
                dX = dxb[n]
                ops.conv3x3_dgrad(draw, self.w_dgrad[n], dX)
                if b is not None:                       # concat [up, skip]
                    c0 = act[a].shape[3]
                    skip_grad[b] = (dX, blk.cin, c0)
                    if a in self._ups:                  # through the dropout + nearest upsampling to the previous block
                        ops.upsample2x_bwd(dX, blk.cin, 0, dxb[a], self._dropout_p(a, dropout), seed_base, seed_dev, layer_id[a])
                        grad_of[self._ups[a]] = (dxb[a], c0, 0)
                    else:
                        grad_of[a] = (dX, blk.cin, 0)
                elif a.startswith('pool'):
                    l = int(a[4:])
                    enc = 'enc%db' % l
                    sg, lds, offs = skip_grad[enc]
                    out = dxb['skip%d' % l]
                    ops.pool_bwd_add(sg, lds, offs, act[enc], act[a], dX, out)
                    grad_of[enc] = (out, out.shape[3], 0)
                else:
                    grad_of[a] = (dX, blk.cin, 0)
            else:
                on_wgrad_stream(ops.convT2x2_wgrad, act[a], draw, self.G[n + '/kernel'], s['wgrad_ws'])
                dX = dxb[n]
                ops.convT2x2_dgrad(draw, self.w_dgrad[n], dX)
                grad_of[a] = (dX, blk.cin, 0)
        if side is not None:                            # join: every weight gradient is complete before the optimizer
            ev = torch.cuda.Event()
            ev.record(side)
            main.wait_event(ev)
        # ---------------- data-parallel: gradient of the global-batch loss (NCCL all-reduce of the flat 31 MB buffer).
        # It runs AFTER the backward pass on purpose: the single-launch BatchNorm kernels spin on peers' flags while they
        # hold their SMs, and an NCCL kernel that needs SMs on this rank while its partner waits behind such a kernel on
        # the other rank would close a dependency cycle.  Only the (non-blocking) weight-gradient kernels ever run
        # concurrently with the spinning kernels.
        self._allreduce(self.grads)
        # ---------------- Keras-form Adam over the flat parameter buffer
        ops.adam_step(self.params, self.grads, self.adam_m, self.adam_v, 0., self.lr_t, beta1, beta2, eps)

    @_on_engine_device
    def train_step(self, x_dev, y_dev, loss='dice_loss', lr=0.002, dropout=True, beta1=0.9, beta2=0.999, eps=1e-8):
        """One train_on_batch.  x_dev fp32 [B,h,w], y_dev uint8 [B,h,w] on the device.
        Returns the device tensor [loss, F1, prec, reca, dice, dicesq, posyt, posyp] (static buffer)."""
        if self.dtype == torch.float16:
            raise ValueError("precision 'fp16' is inference only (gradients underflow in fp16); train in 'bf16' or 'fp32'")
        B, H, W = x_dev.shape
        s = self._session(B, H, W, True)
        s['x'].copy_(x_dev)
        s['y'].copy_(y_dev)
        loss_id = nat.LOSS_IDS[loss] if isinstance(loss, str) else int(loss)
        key = ('train', loss_id, float(lr), bool(dropout), beta1, beta2, eps)
        # the weights-as-M orientation of the generic kernel pays on the 512^2 inference shapes but not on the small
        # images of a training crop (profiles/r2_swap_sweep.txt): pinned off while the step is enqueued / captured
        # Programmatic dependent launch along the main chain is available (pdl_train; the conv / dgrad kernels read only the
        # step's static data before their dependency wait, the BatchNorm / pooling kernels wait at entry) but off by default,
        # see __init__.  Cross-stream edges (the weight-gradient side stream) are ordinary full dependencies either way.
        def enqueue():
            with nat.policy(swap_min_cout=0, pdl=1 if self.pdl_train else 0):
                self._train_step_enqueue(s, loss_id, lr, dropout, beta1, beta2, eps)
        self._run_graphed(s['tta_graphs'], key, enqueue)
        self.iteration += 1
        self._weights_dirty = True
        return self.metrics
