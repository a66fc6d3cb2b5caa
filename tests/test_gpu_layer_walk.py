"""Teacher-forced layer walk through the inference engine: every layer of an eager UNetEngine.infer is checked against
its own float64 rounding bound (tests/rounding_bound.py), with the input the engine actually stored for it.  No error
carries over from earlier layers, so each kernel is held to its own rounding, not to the network's drift.

- conv3x3 / concat / convT: within the bound (16-bit: RN16 of [v - d, v + d]; fp32 check mode: [v - d, v + d]), and
  in every 16-bit tensor at least rounding_bound.EXACT_MIN of the non-zero outputs exactly RN16(v).
- pool<l> (fused into the encoder convs) and upsample2x: bit-equal to the 2x2 max / nearest 2x of the stored tensor.
- dec0b + head (the activation is never stored): the logit within the interval the dec0b bound gives through
  w1 - w0 of the head, and prob = sigmoid(logit) within the error of the kernel's __expf.
- the prepared operands: w_fwd bit-equal to round-to-nearest of the fp32 master weights in the kernel layouts,
  inf_scale / inf_shift the float64 BatchNorm fold within a few fp32 ulps.

The float64 references run on the GPU (torch conv2d / conv_transpose2d in float64)."""
import collections

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import oracle
import rounding_bound as rb

pytestmark = pytest.mark.gpu

MATRIX = ([(p, nfb, mode, (8, 512, 512)) for p in ('fp16', 'bf16') for nfb in (8, 16, 24, 32, 48, 64)
           for mode in ('transpose', 'upsampling')]
          + [('fp32', nfb, mode, (8, 512, 512)) for nfb in (8, 32) for mode in ('transpose', 'upsampling')]
          # a tile width that is not a power of two: level widths 640 / 320 / 160 / 80 / 40
          + [('fp16', nfb, mode, (8, 640, 640)) for nfb in (32, 64) for mode in ('transpose', 'upsampling')])
REACHED = collections.defaultdict(set)       # (precision, nfb) -> kernels the default dispatch ran
DONE = set()

D64 = torch.float64
# __expf: at most 2 + floor(1.173 |x|) ulps (CUDA C Programming Guide, intrinsic functions); 1 + e and the division
# round once each
def _sigmoid_tol(z, p):
    r = (2.0 + torch.floor(1.173 * z.abs())) * 2.0 ** -23
    return p * (1 - p) * r + 4 * rb.U24 * p + 1e-30


def _nchw(t):
    return t.permute(0, 3, 1, 2).to(D64)


def _nhwc(t):
    return t.permute(0, 2, 3, 1)


def _conv_w(eng, blk):
    """the conv3x3 weights the kernel read, as a float64 [Cout, Cin, 3, 3] tensor"""
    w = eng.w_fwd[blk.name]
    if w.dtype == torch.float32:                                    # fp32 master, Keras HWIO (check mode and enc0a)
        return w.view(3, 3, blk.cin, blk.cout).permute(3, 2, 0, 1).to(D64)
    return w.view(blk.cout, 3, 3, blk.cin).permute(0, 3, 1, 2).to(D64)   # [Cout][9][Cin]


def _convT_w(eng, blk):
    """the convT weights the kernel read, as a float64 [Cin, Cout, 2, 2] tensor"""
    w = eng.w_fwd[blk.name]
    if w.dtype == torch.float32:                                    # fp32 layout [4][Cin][Cout]
        return w.view(2, 2, blk.cin, blk.cout).permute(2, 3, 0, 1).to(D64)
    return w.view(2, 2, blk.cout, blk.cin).permute(3, 2, 0, 1).to(D64)   # [4][Cout][Cin]


def _bits_equal(a, b):
    """bit-equal 16-bit / fp32 tensors (a max over +0 and -0 may return either zero)"""
    assert a.dtype == b.dtype and a.shape == b.shape
    it = {2: torch.int16, 4: torch.int32}[a.element_size()]
    return bool(((a.view(it) == b.view(it)) | ((a == 0) & (b == 0))).all())


def _check_prepared(eng):
    for blk in eng.dspec.blocks:
        if blk.kind == 'head':
            continue
        n = blk.name
        k = eng.P[n + '/kernel']
        wf = eng.w_fwd[n]
        if wf.dtype != torch.float32:
            want = (k.permute(3, 0, 1, 2) if blk.kind == 'conv' else k).reshape(-1).to(wf.dtype)
            assert _bits_equal(wf, want), '%s: w_fwd is not RN16 of the master weights' % n
        elif blk.kind == 'up':
            assert torch.equal(wf, k.permute(0, 1, 3, 2).reshape(-1)), n
        P = {p: eng.P['%s/%s' % (n, p)].to(D64) for p in ('gamma', 'beta', 'moving_mean', 'moving_var', 'bias')}
        s = P['gamma'] / torch.sqrt(P['moving_var'] + float(np.float32(1e-3)))
        t = P['beta'] + (P['bias'] - P['moving_mean']) * s
        sc, sh = eng.inf_scale[n].to(D64), eng.inf_shift[n].to(D64)
        assert bool(((sc - s).abs() <= 4 * rb.U24 * s.abs()).all()), '%s: folded scale' % n
        mag = P['beta'].abs() + ((P['bias'] - P['moving_mean']) * s).abs()
        assert bool(((sh - t).abs() <= 6 * rb.U24 * mag + 1e-30).all()), '%s: folded shift' % n


def _record_kernels(monkeypatch, precision):
    """wrap the engine's contraction calls: output tensor address -> the kernel the call dispatched to"""
    from deepcalcium import _native as nat
    from deepcalcium.engine import ops
    log = {}
    for name, out_arg in (('conv3x3_fwd', 3), ('conv3x3_fwd_fused', 3), ('conv3x3_c1_fwd', 2), ('convT2x2_fwd', 2)):
        fn = getattr(ops, name)

        def wrapped(*a, _fn=fn, _name=name, _o=out_arg, **k):
            _fn(*a, **k)
            if _name == 'conv3x3_c1_fwd':
                kern = 'c1'
            elif precision == 'fp32':
                kern = 'f32'
            else:
                kern = nat.last_kernel() + ('+head' if k.get('head_kernel') is not None else '')
            log[a[_o].data_ptr()] = kern
        monkeypatch.setattr(ops, name, wrapped)
    return log


def _layer_reference(eng, s, blk):
    """(A, B) in float64 NHWC from the stored inputs of block blk"""
    act = s['act']
    a, b = eng._inputs[blk.name]
    if blk.kind == 'up':
        x = _nchw(act[a])
        w = _convT_w(eng, blk)
        A = F.conv_transpose2d(x, w, stride=2)
        B = F.conv_transpose2d(x.abs(), w.abs(), stride=2)
    else:
        if blk.cin == 1:
            x = s['x'][:, None].to(D64)
        else:
            x = _nchw(act[a]) if b is None else torch.cat([_nchw(act[a]), _nchw(act[b])], 1)
        w = _conv_w(eng, blk)
        A = F.conv2d(x, w, padding=1)
        B = F.conv2d(x.abs(), w.abs(), padding=1)
    return _nhwc(A), _nhwc(B)


def _c_acc(eng, blk):
    if blk.cin == 1:                  # K = 9 with fp32 products (the c1 kernel, and the fp32 check mode's enc0a)
        return rb.C_ACC_C1
    return rb.C_ACC_F32 if eng.precision == 'fp32' else rb.c_acc_tc(blk.cin * (9 if blk.kind == 'conv' else 1))


@pytest.mark.parametrize('point', MATRIX, ids=['%s-nfb%d-%s-%dx%dx%d' % ((p, n, m) + s) for p, n, m, s in MATRIX])
def test_every_layer_within_its_rounding_bound(cuda, monkeypatch, point):
    from deepcalcium.engine.graph import GraphSpec
    from deepcalcium.engine.unet_engine import UNetEngine
    precision, nfb, mode, shape = point
    log = _record_kernels(monkeypatch, precision)
    eng = UNetEngine(GraphSpec(nfb, upsampling_or_transpose=mode), precision=precision, use_graphs=False)
    eng.set_weights_dict(oracle.init_weights(oracle.UNetSpec(nfb, upsampling_or_transpose=mode), seed=100 + nfb))
    x = torch.from_numpy(np.random.default_rng(nfb).standard_normal(shape).astype(np.float32)).cuda()
    prob, logit = eng.infer(x)
    torch.cuda.synchronize()
    _check_prepared(eng)
    s = eng._sessions[(shape[0], shape[1], shape[2], False)]
    act = s['act']
    rows = []
    for blk in eng.dspec.blocks:
        n = blk.name
        if blk.kind == 'head':
            continue
        a, _ = eng._inputs[n]
        if a in eng._ups:                                           # nearest 2x of the stored tensor, bit for bit
            src = act[eng._ups[a]]
            want = src.repeat_interleave(2, 1).repeat_interleave(2, 2)
            assert _bits_equal(act[a], want), '%s: upsample2x' % a
        A, B = _layer_reference(eng, s, blk)
        sc, sh = eng.inf_scale[n].to(D64), eng.inf_shift[n].to(D64)
        kern = log.get(act[n].data_ptr(), '?')
        c_acc = _c_acc(eng, blk)
        if n == 'dec0b':
            rep = _check_head(eng, s, A, B, sc, sh, c_acc, prob, logit)
        else:
            rep = rb.check(act[n], A, B, sc, sh, c_acc=c_acc)
            rb.assert_ok(rep, '%s %s (%s)' % (point, n, kern), exact=precision != 'fp32')
        if n in ('enc0b', 'enc1b', 'enc2b', 'enc3b'):              # the pooled copy: 2x2 max of the stored activation
            pool = act['pool%d' % blk.level]
            want = _nhwc(F.max_pool2d(act[n].permute(0, 3, 1, 2).float(), 2)).to(pool.dtype)
            assert _bits_equal(pool, want.contiguous()), '%s: pool%d' % (n, blk.level)
        rows.append((n, kern, rep))
        REACHED[(precision, nfb)].add(kern)
        del A, B
    DONE.add(point)
    print('\n%s' % (point,))
    print('  %-6s %-26s %9s %9s %9s %10s %8s' % ('layer', 'kernel', 'exact', 'exact nz', 'max ulp', 'med d ulp', 'sharp'))
    for n, kern, rep in rows:
        print('  %-6s %-26s %9.6f %9.6f %9.3g %10.3g %8.5f' % (n, kern, rep['exact'], rep['exact_nz'], rep['max_ulp'],
                                                                rep['median_delta_ulp'], rep['sharp']))


def _check_head(eng, s, A, B, sc, sh, c_acc, prob, logit):
    """dec0b is never stored (need_y=False): the kernel sums y_c * (w1 - w0)_c in fp32, with y_c the activation
    either rounded to the 16-bit format or left in fp32 (the fused epilogue need not round what it does not store).
    The logit lies in the interval those admissible y_c give, widened by the fp32 summation error of the C-term head
    dot product."""
    fmt = rb.TORCH_FORMAT[eng.dtype]
    v = sc * A + sh
    d = rb.delta(A, B, sc, sh, c_acc)
    lo, hi = rb.interval(v, d, fmt, relu=True)
    lo = torch.minimum(lo, torch.clamp(v - d, min=0))
    hi = torch.maximum(hi, torch.clamp(v + d, min=0))
    hk = eng.P['head/kernel'].view(-1, 2)
    wd = (hk[:, 1] - hk[:, 0]).to(D64)                               # formed in fp32, as the kernel does
    hb = float((eng.P['head/bias'][1] - eng.P['head/bias'][0]).item())
    zlo = torch.minimum(lo * wd, hi * wd).sum(-1) + hb
    zhi = torch.maximum(lo * wd, hi * wd).sum(-1) + hb
    C = wd.numel()
    err = (C + 2) * rb.U24 * (torch.maximum(lo.abs(), hi.abs()) * wd.abs()).sum(-1) + 2 * rb.U24 * abs(hb)
    z = logit.to(D64)
    bad = int(((z < zlo - err) | (z > zhi + err) | ~torch.isfinite(z)).sum())
    if bad:
        i = int(((z < zlo - err) | (z > zhi + err) | ~torch.isfinite(z)).reshape(-1).nonzero()[0])
        f = lambda t: float(t.reshape(-1)[i])
        raise AssertionError('dec0b + head: %d logits outside the bound, first z %r in [%r, %r] +- %r, hb %r'
                             % (bad, f(z), f(zlo), f(zhi), f(err), hb))
    p = torch.sigmoid(z)
    pe = (prob.to(D64) - p).abs()
    assert bool((pe <= _sigmoid_tol(z, p)).all()), 'prob vs sigmoid(logit): %g' % float(pe.max())
    # report in the terms of the other layers: the logit's admissible width against its own fp32 ulp
    zr = hb + (torch.clamp(v, min=0) if fmt == 'fp32' else rb.rn(torch.clamp(v, min=0), fmt)) @ wd
    q = rb.quantum(zr, 'fp32')
    ex = float((z == zr.float().double()).double().mean())
    return dict(n=z.numel(), bad=bad, exact=ex, exact_nz=ex,
                max_ulp=float(((z - zr).abs() / q).max()), median_delta_ulp=float(((zhi - zlo + 2 * err) / q).median()),
                sharp=float('nan'))


def test_matrix_reached_kernels():
    """which kernels the default inference dispatch ran over the whole matrix (needs the full matrix in this session)"""
    if len(DONE) < len(MATRIX):
        pytest.skip('the full layer-walk matrix did not run in this session')
    for key in sorted(REACHED):
        print('%s nfb %d: %s' % (key[0], key[1], sorted(REACHED[key])))
    tc = set().union(*(REACHED[k] for k in REACHED if k[0] != 'fp32'))
    print('16-bit kernels reached: %s' % sorted(tc))
    # what the default inference dispatch runs over the matrix (every other variant is reached through forced policies in
    # tests/test_gpu_ops.py): flat only from nfb 48, strip_fold_nsplit_cluster from nfb 16
    assert tc == {'c1', 'flat', 'generic', 'generic_pool', 'generic_swap', 'strip', 'strip_fold', 'strip_fold_fused',
                  'strip_fold_fused+head', 'strip_fold_nsplit_cluster'}, sorted(tc)
