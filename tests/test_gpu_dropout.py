"""Dropout on the GPU against its host statement (tests/dropout_mask.py) and against float64.

Every kernel that draws the keep mask - the separate BatchNorm passes, the single-launch grid-barrier and channel-slab
kernels (with and without the fused 2x2 max-pool), the apply pass from conv-epilogue sums, and the nearest upsampling of
the 'upsampling' graph - is held to the statement bit for bit on a constant input, and to a float64 reference on random
inputs, forward and backward.  The factored softmax-head gradient is checked at the kernel level.  Whole training steps
with dropout on, eager and graph-replayed, are compared with oracle.train_step given the masks the statement says the
engine drew."""
import hashlib

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import dropout_mask as dm
import oracle
from oracle import losses as ol

pytestmark = pytest.mark.gpu

DT = {'fp32': torch.float32, 'bf16': torch.bfloat16}
EPS = 1e-3
SEED = 0x1234567887654321                 # both 32-bit halves nonzero
SEED_DEV = 0x0F1E2D3C4B5A6978
SEED_MODES = ['host', 'device']
MODES = ('transpose', 'upsampling')

# (N, H, W, C): the VEC = 4 paths (C = 4 - the nb_filters_base 4 network's up0 - and 12), M * C not a multiple of 8,
# odd N, C = 32 ... 512, and the levels of a 32 x 128^2 training step (where the channel-slab kernels run)
SHAPES = [(1, 5, 7, 4), (3, 6, 10, 4), (1, 3, 5, 12), (2, 4, 6, 12), (3, 6, 10, 32), (4, 32, 32, 64), (1, 4, 6, 96),
          (5, 12, 20, 128), (3, 8, 8, 512), (32, 128, 128, 32), (32, 64, 64, 64), (32, 32, 32, 128), (32, 16, 16, 256),
          (32, 8, 8, 512)]


def _ids(shapes):
    return ['x'.join(str(v) for v in s) for s in shapes]


def tol(precision, scale=1.0):
    """test_gpu_ops.py's per-precision tolerance"""
    return dict(fp32=2e-4, bf16=3e-2)[precision] * scale


def _draw(shape, seed_mode):
    """(p, layer id, host seed, device seed tensor or None, the seed the kernels draw with) of a case"""
    i = SHAPES.index(shape) if shape in SHAPES else len(shape) + sum(shape)
    p = (0.25, 0.5)[i % 2]
    layer = 17 + i
    if seed_mode == 'host':
        return p, layer, SEED, None, SEED
    seed_dev = torch.tensor([SEED_DEV], dtype=torch.int64, device='cuda')
    return p, layer, SEED, seed_dev, SEED ^ SEED_DEV


def _keep(seed, layer, shape, p, device='cuda'):
    """the statement's fp32 keep scale of an NHWC tensor, on the device"""
    return torch.from_numpy(np.array(dm.keep_scale(seed, layer, int(np.prod(shape)), p))).view(*shape).to(device)


def _coefficients(x, gamma, beta):
    """float64 batch statistics of x [M, C] and the fp32 coefficients a BatchNorm kernel derives from them"""
    x64 = x.double().reshape(-1, x.shape[-1])
    mean = x64.mean(0)
    var = ((x64 - mean) ** 2).mean(0)
    rstd = torch.rsqrt(var + EPS)
    scale = (gamma.double() * rstd).float()
    shift = (beta.double() - mean * scale.double()).float()
    return mean, var, scale, shift, mean.float(), rstd.float()


def _pool(t):
    """2x2 max-pool of an NHWC tensor"""
    return F.max_pool2d(t.permute(0, 3, 1, 2), 2).permute(0, 2, 3, 1)


def _forward_variants(x, gamma, beta, p, seed, seed_dev, layer):
    """run every forward kernel that draws the mask on x [N, H, W, C]: -> [(variant, kernel name, y, pooled copy)]; a
    variant that rejects the shape (DcbError) is listed with kernel None"""
    from deepcalcium import _native as nat
    from deepcalcium.engine import ops
    N, H, W, C = x.shape
    M = N * H * W
    f = lambda: torch.empty(C, device='cuda')
    mm = lambda: torch.zeros(C, device='cuda')
    mv = lambda: torch.ones(C, device='cuda')
    x64 = x.double().reshape(M, C)
    sums = torch.cat([x64.sum(0), (x64 * x64).sum(0)]).contiguous()
    sums_q = torch.round(sums * 2 ** 20).to(torch.int64).contiguous()
    _, _, scale, shift, _, _ = _coefficients(x, gamma, beta)
    pools = (False, True) if H % 2 == 0 and W % 2 == 0 else (False,)
    out = []

    def run(variant, fn, pooled=False, **pol):
        y = torch.empty_like(x)
        pl = torch.empty(N, H // 2, W // 2, C, dtype=x.dtype, device='cuda') if pooled else None
        try:
            with nat.policy(**pol):
                fn(y, pl)
            kernel = nat.last_kernel()
        except nat.DcbError:
            out.append((variant, None, None, None))
            return
        torch.cuda.synchronize()
        if pol.get('bn_slab') == 0:
            assert not kernel.startswith('bn_slab'), (variant, kernel)
        out.append((variant, kernel, y, pl))

    run('bn_apply', lambda y, pl: ops.bn_apply(x, scale, shift, y, True, p, seed, seed_dev, layer))
    run('bn_finalize_apply', lambda y, pl: ops.bn_finalize_apply(x, sums, M, gamma, beta, 0.99, mm(), mv(), f(), f(), f(), f(),
                                                                 y, True, p, seed, seed_dev, layer))
    for pooled in pools:
        for slab in (0, 1, 2):
            def fwd(y, pl):
                ws = torch.zeros(ops.bn_train_workspace_bytes(C), dtype=torch.uint8, device='cuda')
                sync = torch.zeros(4, dtype=torch.int32, device='cuda')
                ops.bn_train_fwd(x, gamma, beta, 0.99, mm(), mv(), f(), f(), f(), f(), y, ws, sync, True, p, seed, seed_dev,
                                 layer, pool_out=pl)
            run('bn_train_fwd slab=%d%s' % (slab, ' pool' if pooled else ''), fwd, pooled, bn_slab=slab)
        run('bn_train_fwd_sums%s' % (' pool' if pooled else ''),
            lambda y, pl: ops.bn_train_fwd_sums(x, sums_q, gamma, beta, 0.99, mm(), mv(), f(), f(), f(), f(), y, True, p, seed,
                                                seed_dev, layer, pool_out=pl), pooled)
    return out


@pytest.mark.parametrize('seed_mode', SEED_MODES)
@pytest.mark.parametrize('precision', ['fp32', 'bf16'])
@pytest.mark.parametrize('shape', SHAPES, ids=_ids(SHAPES))
def test_forward_mask_bit_for_bit(cuda, shape, precision, seed_mode):
    """constant input, gamma 0, beta 1 (bn_apply: scale 0, shift 1): every element is relu(1) * keep, i.e. exactly the
    keep scale rounded to the stored dtype; a pooled copy is exactly the max-pool of the stored values"""
    dt = DT[precision]
    p, layer, seed, seed_dev, eff = _draw(shape, seed_mode)
    N, H, W, C = shape
    x = torch.ones(shape, dtype=dt, device='cuda')
    want = _keep(eff, layer, shape, p).to(dt)
    ran = []
    for variant, kernel, y, pl in _forward_variants(x, torch.zeros(C, device='cuda'), torch.ones(C, device='cuda'), p, seed,
                                                    seed_dev, layer):
        if kernel is None:
            continue
        assert torch.equal(y, want), (variant, kernel)
        if pl is not None:
            assert torch.equal(pl, _pool(y.float()).to(dt)), (variant, kernel)
        ran.append('%s -> %s' % (variant, kernel))
    print('%s %s: %s' % (precision, shape, '; '.join(ran)))
    assert ran


@pytest.mark.parametrize('seed_mode', SEED_MODES)
@pytest.mark.parametrize('precision', ['fp32', 'bf16'])
@pytest.mark.parametrize('shape', SHAPES, ids=_ids(SHAPES))
def test_forward_values_against_float64(cuda, shape, precision, seed_mode):
    """random x: y = relu(BN(x)) * keep against float64 (the tolerance of test_batchnorm_train_forward_backward); a pooled
    copy is exactly the max-pool of the stored values and within the same tolerance of the float64 pool"""
    dt = DT[precision]
    p, layer, seed, seed_dev, eff = _draw(shape, seed_mode)
    N, H, W, C = shape
    rng = np.random.default_rng(sum(shape))
    x = torch.from_numpy(rng.standard_normal(shape) * 2 + 0.5).to(dt).cuda()
    gamma = torch.from_numpy(rng.uniform(0.5, 1.5, C)).float().cuda()
    beta = torch.from_numpy(0.1 * rng.standard_normal(C)).float().cuda()
    mean, var, _, _, _, _ = _coefficients(x, gamma, beta)
    z = (x.double() - mean) * torch.rsqrt(var + EPS) * gamma.double() + beta.double()
    ref = torch.relu(z) * _keep(eff, layer, shape, p).double()
    for variant, kernel, y, pl in _forward_variants(x, gamma, beta, p, seed, seed_dev, layer):
        if kernel is None:
            continue
        err = float((y.double() - ref).abs().max())
        assert err < tol(precision, 4), (variant, kernel, err)
        if pl is not None:
            assert torch.equal(pl, _pool(y.float()).to(dt)), (variant, kernel)
            assert float((pl.double() - _pool(ref)).abs().max()) < tol(precision, 4), (variant, kernel)


def _backward_reference(x, gamma, beta, scale, shift, keep, dy):
    """float64 autograd of relu(BN(x)) * keep with batch statistics.  The ReLU gate is taken where the kernels take it,
    at x * scale + shift > 0 with the fp32 coefficients they are given (evaluated exactly: the fp32 product is exact in
    float64, so the sign of the float64 sum is the sign of the kernels' fused multiply-add); a float64 gate would flip the
    few elements within an fp32 rounding of 0, each by a whole gradient value."""
    C = x.shape[-1]
    x64 = x.double().reshape(-1, C).clone().requires_grad_(True)
    g64 = gamma.double().clone().requires_grad_(True)
    b64 = beta.double().clone().requires_grad_(True)
    mean = x64.mean(0)
    var = ((x64 - mean) ** 2).mean(0)
    z = (x64 - mean) * torch.rsqrt(var + EPS) * g64 + b64
    gate = (x64.detach() * scale.double() + shift.double() > 0).double()
    (z * gate * keep.double().reshape(-1, C)).backward(dy)
    return x64.grad, g64.grad, b64.grad


def _assert_backward(precision, what, draw, dg, db, ref):
    gx, gg, gb = ref
    t = tol(precision, 4)
    err = float((draw.double().reshape(gx.shape) - gx).abs().max())
    assert err < t, (what, err)
    rt = 1e-2 if precision == 'bf16' else 1e-4
    assert torch.allclose(dg.double(), gg, atol=t * 30, rtol=rt), (what, float((dg.double() - gg).abs().max()))
    assert torch.allclose(db.double(), gb, atol=t * 30, rtol=rt), (what, float((db.double() - gb).abs().max()))


@pytest.mark.parametrize('seed_mode', SEED_MODES)
@pytest.mark.parametrize('precision', ['fp32', 'bf16'])
@pytest.mark.parametrize('shape', SHAPES, ids=_ids(SHAPES))
def test_backward_against_float64(cuda, shape, precision, seed_mode):
    """draw, dgamma, dbeta of bn_bwd_reduce + bn_bwd_apply and of bn_train_bwd (grid-barrier and channel-slab kernels), dy
    a channel slice of a wider fp32 tensor (ldy = 2C, offy = C/2), against float64 autograd of relu(BN(x)) * keep"""
    from deepcalcium import _native as nat
    from deepcalcium.engine import ops
    dt = DT[precision]
    p, layer, seed, seed_dev, eff = _draw(shape, seed_mode)
    N, H, W, C = shape
    M = N * H * W
    rng = np.random.default_rng(sum(shape) + 1)
    x = torch.from_numpy(rng.standard_normal(shape) * 2 + 0.5).to(dt).cuda()
    gamma = torch.from_numpy(rng.uniform(0.5, 1.5, C)).float().cuda()
    beta = torch.from_numpy(0.1 * rng.standard_normal(C)).float().cuda()
    _, _, scale, shift, mean32, rstd32 = _coefficients(x, gamma, beta)
    dy_wide = torch.from_numpy(rng.standard_normal((M, 2 * C))).float().cuda()
    off = C // 2 if (C // 2) % 4 == 0 else 0
    ref = _backward_reference(x, gamma, beta, scale, shift, _keep(eff, layer, shape, p), dy_wide[:, off:off + C].double())
    f = lambda: torch.empty(C, device='cuda')
    ran = []
    draw, dg, db = torch.empty_like(x), f(), f()
    sums = torch.zeros(2 * C, dtype=torch.float64, device='cuda')
    try:
        ops.bn_bwd_reduce(dy_wide, 2 * C, off, x, scale, shift, mean32, rstd32, sums, p, seed, seed_dev, layer)
        k_reduce = nat.last_kernel()
        ops.bn_bwd_apply(dy_wide, 2 * C, off, x, scale, shift, mean32, rstd32, sums, draw, dg, db, p, seed, seed_dev, layer)
        torch.cuda.synchronize()
        _assert_backward(precision, 'bn_bwd_reduce + bn_bwd_apply', draw, dg, db, ref)
        ran.append('%s + %s' % (k_reduce, nat.last_kernel()))
    except nat.DcbError:
        pass
    for slab in (0, 1, 2):
        draw, dg, db = torch.empty_like(x), f(), f()
        ws = torch.zeros(ops.bn_train_workspace_bytes(C), dtype=torch.uint8, device='cuda')
        sync = torch.zeros(4, dtype=torch.int32, device='cuda')
        try:
            with nat.policy(bn_slab=slab):
                ops.bn_train_bwd(dy_wide, 2 * C, off, x, scale, shift, mean32, rstd32, draw, dg, db, ws, sync, p, seed, seed_dev,
                                 layer)
            kernel = nat.last_kernel()
        except nat.DcbError:
            continue
        torch.cuda.synchronize()
        assert slab != 0 or not kernel.startswith('bn_slab'), kernel
        _assert_backward(precision, 'bn_train_bwd slab=%d (%s)' % (slab, kernel), draw, dg, db, ref)
        ran.append('slab=%d -> %s' % (slab, kernel))
    print('%s %s: %s' % (precision, shape, '; '.join(ran)))
    assert ran or C in (12, 96)          # C/4 or C/8 must divide 256 for the reducing kernels


# (N, h, w, C, ldy): the input of the 'upsampling' graph's up<l> and the row stride of the concat gradient it reads
UP_SHAPES = [(1, 3, 5, 4, 8), (3, 4, 6, 12, 24), (2, 5, 7, 32, 64), (1, 4, 4, 512, 768), (32, 16, 16, 256, 384)]


@pytest.mark.parametrize('seed_mode', SEED_MODES)
@pytest.mark.parametrize('precision', ['fp32', 'bf16'])
@pytest.mark.parametrize('shape', UP_SHAPES, ids=_ids(UP_SHAPES))
def test_upsample2x_dropout_forward_and_backward(cuda, shape, precision, seed_mode):
    """upsample2x: ones in -> exactly the keep scale; random x -> exactly the fp32 product x * keep, rounded to the dtype.
    upsample2x_bwd (ldy = the concat width, offy = 0, as the engine calls it): against float64 autograd of
    upsample-then-mask within its rounding bound (four fp32 products and three sums: 5 * 2^-24 * sum |terms|), and with
    dy = 1 bit for bit the fp32 sum of the four keep scales in the kernel's order."""
    from deepcalcium.engine import ops
    dt = DT[precision]
    N, h, w, C, ldy = shape
    p, layer, seed, seed_dev, eff = _draw(shape, seed_mode)
    out_shape = (N, 2 * h, 2 * w, C)
    keep = _keep(eff, layer, out_shape, p)
    y = torch.empty(out_shape, dtype=dt, device='cuda')
    ops.upsample2x(torch.ones(N, h, w, C, dtype=dt, device='cuda'), y, p, seed, seed_dev, layer)
    assert torch.equal(y, keep.to(dt))
    rng = np.random.default_rng(sum(shape))
    x = torch.from_numpy(rng.standard_normal((N, h, w, C))).to(dt).cuda()
    ops.upsample2x(x, y, p, seed, seed_dev, layer)
    up = x.float().repeat_interleave(2, dim=1).repeat_interleave(2, dim=2)
    assert torch.equal(y, (up * keep).to(dt))
    # backward
    dy = torch.from_numpy(rng.standard_normal((N, 2 * h, 2 * w, ldy))).float().cuda()
    dx = torch.empty(N, h, w, C, device='cuda')
    ops.upsample2x_bwd(dy, ldy, 0, dx, p, seed, seed_dev, layer)
    xr = torch.zeros(N, h, w, C, dtype=torch.float64, device='cuda', requires_grad=True)
    (xr.repeat_interleave(2, dim=1).repeat_interleave(2, dim=2) * keep.double()).backward(dy[..., :C].double())
    terms = (dy[..., :C].double() * keep.double()).abs()
    bound = 5 * 2.0 ** -24 * terms.view(N, h, 2, w, 2, C).sum(dim=(2, 4))
    assert bool(((dx.double() - xr.grad).abs() <= bound).all())
    ops.upsample2x_bwd(torch.ones(N, 2 * h, 2 * w, ldy, device='cuda'), ldy, 0, dx, p, seed, seed_dev, layer)
    k = keep.view(N, h, 2, w, 2, C)
    acc = torch.zeros(N, h, w, C, device='cuda')
    for a in (0, 1):
        for b in (0, 1):
            acc = acc + k[:, :, a, :, b, :]                    # fp32 adds in the kernel's order
    assert torch.equal(dx, acc)


LOSSES = ['dice_loss', 'binary_crossentropy', 'dicesq_loss', 'weighted_binary_crossentropy']


@pytest.mark.parametrize('precision', ['fp32', 'bf16'])
@pytest.mark.parametrize('loss', LOSSES)
def test_rank1_head_gradient_factors(cuda, loss, precision):
    """head_loss_bwd_rank1 writes gpix[m] and wd[c]: their product is head_loss_bwd's dL/dx bit for bit and within the
    criteria of test_head_loss_metrics_and_gradient of float64 autograd; dw and the metrics are head_loss_bwd's.  M is not a
    multiple of the 256-thread CTA.  Inputs other than 32 channels are rejected."""
    from deepcalcium import _native as nat
    from deepcalcium.engine import ops
    dt = DT[precision]
    rng = np.random.default_rng(17)
    M, C = 3001, 32
    x = torch.from_numpy(rng.standard_normal((M, C))).to(dt)
    w = (rng.standard_normal((C, 2)) * 0.3).astype(np.float32)
    b = np.array([0.1, -0.2], np.float32)
    yt = (rng.random(M) < 0.126).astype(np.uint8)
    xt = x.double().clone().requires_grad_(True)
    p = torch.softmax(xt @ torch.tensor(w, dtype=torch.float64) + torch.tensor(b, dtype=torch.float64), dim=1)[:, -1]
    ol.LOSSES[loss](torch.tensor(yt, dtype=torch.float64), p).backward()
    xd = x.cuda().view(1, 1, M, C)
    wd_, bd, yd = torch.from_numpy(w).cuda(), torch.from_numpy(b).cuda(), torch.from_numpy(yt).cuda()
    prob = torch.empty(M, device='cuda')
    sums = torch.zeros(8, dtype=torch.float64, device='cuda')
    ops.head_loss_fwd(xd, wd_, bd, yd, prob, sums)
    dx = torch.empty(1, 1, M, C, device='cuda')
    dwb0, dwb1 = (torch.zeros(2 * C + 2, dtype=torch.float64, device='cuda') for _ in range(2))
    dw0, dw1 = torch.empty(2 * C + 2, device='cuda'), torch.empty(2 * C + 2, device='cuda')
    met0, met1 = torch.empty(8, device='cuda'), torch.empty(8, device='cuda')
    ops.head_loss_bwd(xd, wd_, yd, prob, sums, nat.LOSS_IDS[loss], dx, dwb0, dw0, met0)
    gpix, wdiff = torch.empty(M, device='cuda'), torch.empty(C, device='cuda')
    ops.head_loss_bwd_rank1(xd, wd_, yd, prob, sums, nat.LOSS_IDS[loss], gpix, wdiff, dwb1, dw1, met1)
    torch.cuda.synchronize()
    outer = gpix[:, None] * wdiff[None, :]
    assert torch.equal(outer, dx.view(M, C))
    gscale = float(xt.grad.abs().max())
    assert float((outer.double().cpu() - xt.grad).abs().max()) < (1e-2 if precision == 'bf16' else 1e-4) * gscale + 1e-9
    assert torch.equal(met1, met0)
    assert torch.allclose(dw1, dw0, rtol=1e-6, atol=1e-7 * float(dw0.abs().max()))
    x64 = torch.from_numpy(rng.standard_normal((M, 64))).to(dt).cuda().view(1, 1, M, 64)
    with pytest.raises(nat.DcbError):
        ops.head_loss_bwd_rank1(x64, torch.zeros(128, device='cuda'), yd, prob, sums, nat.LOSS_IDS[loss], gpix,
                                torch.empty(64, device='cuda'), dwb1, torch.empty(130, device='cuda'), met1)


@pytest.mark.parametrize('seed_mode', SEED_MODES)
@pytest.mark.parametrize('p', [0.0, 0.25])
@pytest.mark.parametrize('precision', ['fp32', 'bf16'])
def test_rank1_batchnorm_backward(cuda, precision, p, seed_mode):
    """bn_train_bwd_rank1 (dy = gpix[m] * wd[c] rebuilt while it reads) against bn_train_bwd on the materialised product -
    the same kernel up to the compiler contracting the product into the multiply-adds that consume it, so within 1e-3
    relative L2 (test_factored_head_gradient_equals_the_materialised_one) - and both against float64 autograd.  p = 0 is the
    engine's case (the last block has no dropout); p = 0.25 draws the mask inside the rank-1 kernel."""
    from deepcalcium import _native as nat
    from deepcalcium.engine import ops
    dt = DT[precision]
    M, C = 3001, 32
    _, layer, seed, seed_dev, eff = _draw((M, C), seed_mode)
    rng = np.random.default_rng(29)
    x = torch.from_numpy(rng.standard_normal((M, C)) * 2 + 0.5).to(dt).cuda()
    gamma = torch.from_numpy(rng.uniform(0.5, 1.5, C)).float().cuda()
    beta = torch.from_numpy(0.1 * rng.standard_normal(C)).float().cuda()
    gpix = torch.from_numpy(rng.standard_normal(M)).float().cuda()
    wd = torch.from_numpy(rng.standard_normal(C)).float().cuda()
    _, _, scale, shift, mean32, rstd32 = _coefficients(x, gamma, beta)
    keep = _keep(eff, layer, (M, C), p) if p > 0 else torch.ones(M, C, device='cuda')
    ref = _backward_reference(x, gamma, beta, scale, shift, keep, gpix.double()[:, None] * wd.double()[None, :])
    outs = {}
    for rank1 in (True, False):
        draw, dg, db = torch.empty_like(x), torch.empty(C, device='cuda'), torch.empty(C, device='cuda')
        ws = torch.zeros(ops.bn_train_workspace_bytes(C), dtype=torch.uint8, device='cuda')
        sync = torch.zeros(4, dtype=torch.int32, device='cuda')
        with nat.policy(bn_slab=0):       # the rank-1 gradient never takes the slab kernel: compare like with like
            if rank1:
                ops.bn_train_bwd_rank1(gpix, wd, x, scale, shift, mean32, rstd32, draw, dg, db, ws, sync, p, seed, seed_dev, layer)
            else:
                dy = (gpix[:, None] * wd[None, :]).contiguous()
                ops.bn_train_bwd(dy, C, 0, x, scale, shift, mean32, rstd32, draw, dg, db, ws, sync, p, seed, seed_dev, layer)
            kernel = nat.last_kernel()
        torch.cuda.synchronize()
        assert kernel == ('bn_train_bwd_v8_rank1' if rank1 else 'bn_train_bwd_v8'), kernel
        _assert_backward(precision, kernel, draw, dg, db, ref)
        outs[rank1] = (draw.double(), dg.double(), db.double())
    for a, b_ in zip(outs[True], outs[False]):
        assert float((a - b_).norm() / (b_.norm() + 1e-30)) < 1e-3


# ---------------------------------------------------------------- whole training steps with dropout on
_ORACLE = {}


def _case(nfb, mode='transpose'):
    spec = oracle.UNetSpec(nfb, upsampling_or_transpose=mode)
    return spec, oracle.init_weights(spec, seed=7535)


def _batch():
    rng = np.random.default_rng(865)
    x = rng.standard_normal((4, 32, 32)).astype(np.float32)
    return x, (rng.random((4, 32, 32)) < 0.126).astype(np.uint8)


def _engine(nfb, precision, w, mode='transpose', **kw):
    from deepcalcium.engine.graph import GraphSpec
    from deepcalcium.engine.unet_engine import UNetEngine
    eng = UNetEngine(GraphSpec(nfb, upsampling_or_transpose=mode), precision=precision, **kw)
    eng.set_weights_dict(w)
    return eng


def _oracle_step(spec, w, x, y, masks, emulate_bf16=False, gates=None):
    """oracle.train_step with the given masks (and ReLU decisions) -> (loss, new weights, gradients); cached: the first
    step of every engine draws with the same device seed, so tests share the float64 runs"""
    arrays = list(masks.values()) + (list(gates.values()) if gates else [])
    digest = hashlib.sha1(b''.join(np.ascontiguousarray(m, np.uint8).tobytes() for m in arrays)).hexdigest()
    key = (spec, emulate_bf16, digest)
    if key not in _ORACLE:
        L, nw, _, g, _ = oracle.train_step(w, x, y, spec=spec, loss='dice_loss', dropout_keep=masks, emulate_bf16=emulate_bf16,
                                           relu_gate=gates)
        _ORACLE[key] = (L, nw, g)
    return _ORACLE[key]


# A pre-activation within this distance of 0 has no sign that every correct fp32 evaluation agrees on: the convolutions
# put ~1e-6 of rounding on these values of order 1, and the first two steps of this network each have such an element
# (2e-7 and 5e-7 from 0 in dec2b).  One ReLU decision flipped there moves every gradient below it by ~1e-2 relative L2.
GATE_TIE = 1e-5


def _relu_gates(eng, spec, w, x, masks):
    """the ReLU decisions of the engine's fp32 step, read from its stored activations, for the oracle to take - after
    checking that they differ from float64's only at pre-activations within GATE_TIE of 0 (elements the mask drops
    have no decision to compare).  -> ({block: 0/1 [N, C, H, W]}, number of decisions that differ)"""
    B, H, W = x.shape
    act = eng._sessions[(B, H, W, True)]['act']
    o = oracle.unet_forward(w, x, spec, training=True, dropout_keep=masks, return_intermediates=True)
    gates, differ_total = {}, 0
    for name, kind, _, _ in spec.blocks():
        if kind == 'head':
            continue
        raw = o['intermediates'][name + '/raw'].detach()
        mean, var = o['bn_stats'][name]
        sc = torch.rsqrt(var + EPS) * torch.as_tensor(w[name + '/gamma'], dtype=torch.float64)
        sh = torch.as_tensor(w[name + '/beta'], dtype=torch.float64)
        z = (raw - mean[None, :, None, None]) * sc[None, :, None, None] + sh[None, :, None, None]
        gate = act[name].float().permute(0, 3, 1, 2).cpu().double() > 0
        differ = gate != (z > 0)
        if name in masks:
            differ &= torch.as_tensor(masks[name]) > 0
        assert bool((z.abs()[differ] < GATE_TIE).all()), (name, float(z.abs()[differ].max()))
        differ_total += int(differ.sum())
        gates[name] = gate.double().numpy()
    return gates, differ_total


def _rel(a, b):
    return np.linalg.norm(a - b) / (np.linalg.norm(b) + 1e-30)


def _grads(eng):
    from deepcalcium.engine.graph import unpack
    return {k: v.astype(np.float64) for k, v in unpack(eng.spec, eng.dspec, {k: t.cpu().numpy() for k, t in eng.G.items()}).items()}


def _errors(grads, g_ref):
    """relative L2 error of every gradient tensor (a conv bias that feeds a batch-statistics BatchNorm has gradient 0)"""
    return {k: _rel(grads[k], r) for k, r in g_ref.items() if not (k.endswith('/bias') and not k.startswith('head'))}


def _moving_keys(mode):
    return ('enc2b/moving_mean', 'dec1a/moving_var', 'up0/moving_var' if mode == 'transpose' else 'dec0a/moving_mean')


@pytest.mark.parametrize('mode', MODES)
@pytest.mark.parametrize('fused_bn', [1, 0])
def test_dropout_train_step_fp32_against_oracle(cuda, fused_bn, mode):
    """fp32 check mode, dice, dropout on, nb_filters_base 32 at 4 x 32 x 32: the criteria of
    test_train_step_nfb32_against_oracle (loss within 1e-4, every gradient tensor within 3e-3 relative L2, the BatchNorm
    moving statistics) against oracle.train_step given the masks the statement says the step drew, and the step's own ReLU
    decisions at pre-activations within GATE_TIE of 0"""
    from deepcalcium import _native as nat
    spec, w = _case(32, mode)
    x, y = _batch()
    eng = _engine(32, 'fp32', w, mode, use_graphs=False)
    with nat.policy(fused_bn=fused_bn):
        m = eng.train_step(torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda(), loss='dice_loss', dropout=True)
    masks = dm.engine_keep_masks(eng, *x.shape)
    gates, ties = _relu_gates(eng, spec, w, x, masks)
    L, nw, g = _oracle_step(spec, w, x, y, masks, gates=gates)
    assert abs(float(m[0].item()) - L) < 1e-4
    errs = _errors(_grads(eng), g)
    worst = max(errs, key=errs.get)
    print('fp32 %s fused_bn=%d, dropout on: worst gradient relative L2 error vs fp64: %s = %.4g (%d ReLU decisions within %g '
          'of 0 differ from float64)' % (mode, fused_bn, worst, errs[worst], ties, GATE_TIE))
    for key, r in errs.items():
        assert r < 3e-3, (key, r)
    new = eng.get_weights_dict()
    for key in _moving_keys(mode):
        assert np.allclose(new[key], nw[key], atol=1e-4), key


@pytest.mark.parametrize('nfb, fused_bn', [(32, None), (32, 3), (16, None)])
def test_dropout_train_step_bf16_against_the_bf16_emulation(cuda, nfb, fused_bn):
    """bf16, dropout on, under the default policy and with every BatchNorm's statistics taken in the conv epilogues
    (fused_bn 3); nb_filters_base 16 draws its masks over padded channels.  The yardstick is the oracle with bf16 storage
    emulated, given the same masks: loss within 2e-3 of float64, every gradient tensor no further from float64 than
    1.5 x the emulation's distance + 0.03, the median over tensors 1.3 x + 0.03 (test_gpu_widths.py), moving statistics
    within 2e-2."""
    from deepcalcium import _native as nat
    spec, w = _case(nfb)
    x, y = _batch()
    eng = _engine(nfb, 'bf16', w, use_graphs=False)
    pol = {} if fused_bn is None else dict(fused_bn=fused_bn)
    with nat.policy(**pol):
        m = eng.train_step(torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda(), loss='dice_loss', dropout=True)
    masks = dm.engine_keep_masks(eng, *x.shape)
    L, nw, g = _oracle_step(spec, w, x, y, masks)
    g_emu = _oracle_step(spec, w, x, y, masks, emulate_bf16=True)[2]
    assert abs(float(m[0].item()) - L) < 2e-3
    errs = _errors(_grads(eng), g)
    errs_emu = _errors(g_emu, g)
    for key in errs:
        print('nfb %d fused_bn %s %-18s gradient rel. L2 error vs fp64: GPU %.4f, bf16 emulation %.4f'
              % (nfb, fused_bn, key, errs[key], errs_emu[key]))
        assert errs[key] <= 1.5 * errs_emu[key] + 0.03, (key, errs[key], errs_emu[key])
    assert np.median(list(errs.values())) <= 1.3 * np.median(list(errs_emu.values())) + 0.03
    new = eng.get_weights_dict()
    for key in _moving_keys('transpose'):
        assert np.allclose(new[key], nw[key], atol=2e-2), key


def test_dropout_mask_is_fresh_every_step_under_graph_replay(cuda):
    """Three lr = 0 steps (the weights stay put) of a graph-using fp32 engine: eager, capture + replay, replay.  Each step's
    device seed is the previous one advanced by 0x9E3779B97F4A7C15, consecutive steps draw different masks in every
    dropped-out tensor, and each step's loss and gradients meet the fp32 criteria against the oracle given that step's own
    masks (and its own ReLU decisions within GATE_TIE of 0).  Negative control: step 1's gradients against the oracle given
    step 2's masks miss the criterion by more than
    10x - the comparison sees a wrong mask."""
    spec, w = _case(32)
    x, y = _batch()
    xd, yd = torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda()
    eng = _engine(32, 'fp32', w, use_graphs=True)
    steps = []
    for k in range(3):
        m = eng.train_step(xd, yd, loss='dice_loss', lr=0.0, dropout=True)
        assert int(eng.step_state[1].item()) & (2 ** 64 - 1) == (k + 1) * 0x9E3779B97F4A7C15 % 2 ** 64
        masks = dm.engine_keep_masks(eng, *x.shape)
        steps.append((float(m[0].item()), masks, _grads(eng), _relu_gates(eng, spec, w, x, masks)[0]))
    refs = [_oracle_step(spec, w, x, y, masks, gates=gates) for _, masks, _, gates in steps]
    for k, ((loss, masks, grads, _), (L, _, g)) in enumerate(zip(steps, refs)):
        assert abs(loss - L) < 1e-4, (k, loss, L)
        errs = _errors(grads, g)
        assert max(errs.values()) < 3e-3, (k, max(errs, key=errs.get), max(errs.values()))
    for k in (0, 1):
        for name in steps[k][1]:
            assert not np.array_equal(steps[k][1][name], steps[k + 1][1][name]), (k, name)
    wrong = _errors(steps[0][2], refs[1][2])
    worst = max(wrong, key=wrong.get)
    print('negative control: step 1 gradients against the oracle with step 2 masks: worst %s = %.4g, %.0fx the 3e-3 criterion'
          % (worst, wrong[worst], wrong[worst] / 3e-3))
    assert wrong[worst] > 10 * 3e-3
