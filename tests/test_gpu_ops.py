"""Per-kernel parity on the GPU through the C ABI (deepcalcium.engine.ops) against float64 CPU
references built from the oracle's layer arithmetic (torch CPU + autograd).
fp32 = CUDA-core check kernels (tolerance 1e-4 class); bf16 / fp16 = tcgen05 kernels, whose contractions are held to the
float64 rounding bound of tests/rounding_bound.py."""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import oracle
import rounding_bound as rb
from oracle import losses as ol

pytestmark = pytest.mark.gpu

DT = {'fp32': torch.float32, 'bf16': torch.bfloat16, 'fp16': torch.float16}


def dev(a, dtype=torch.float32):
    return torch.as_tensor(np.ascontiguousarray(a)).to(dtype).cuda().contiguous()


def q(a, precision):
    """round an input through the activation dtype so the reference sees the same operand values"""
    t = torch.as_tensor(np.asarray(a, dtype=np.float32))
    return t.to(DT[precision]).to(torch.float64).numpy()


def tol(precision, scale=1.0):
    return dict(fp32=2e-4, bf16=3e-2, fp16=3e-2)[precision] * scale


def nhwc_to_nchw(a):
    return torch.as_tensor(a).permute(0, 3, 1, 2).contiguous()


def assert_bound(got_nchw, A, B, scale, shift, precision, what, c_acc=rb.C_ACC_TC, relu=True):
    """16-bit forward output (NCHW, stored dtype) within its float64 rounding bound (tests/rounding_bound.py)"""
    s = None if scale is None else torch.as_tensor(np.asarray(scale, np.float64))[None, :, None, None]
    t = None if shift is None else torch.as_tensor(np.asarray(shift, np.float64))[None, :, None, None]
    r = rb.check(got_nchw, A.detach(), B.detach(), s, t, c_acc=c_acc, relu=relu, fmt=precision)
    rb.assert_ok(r, what)
    return r


def assert_acc(got, A, B, c_acc, what):
    """fp32 output of a 16-bit contraction (dgrad / wgrad): |y - A| <= c_acc * 2^-24 * B"""
    r = rb.acc_ratio(got, A.detach(), B.detach())
    assert r <= c_acc, '%s: |y - A| = %.3g x 2^-24 B, above c_acc %g' % (what, r, c_acc)
    return r


# Dispatch variants of the bf16 contraction kernels, pinned per call with dcb_set_policy (deepcalcium._native.policy):
# every conv case runs under the DEFAULT policy (what bench.py and smoke() time) and under each forced variant; a
# variant a shape is not eligible for falls through to the next kernel of the dispatch chain, which is checked as well.
FWD_VARIANTS = [
    ('default', {}),
    ('generic', dict(strip=0, flat=0, swap_min_cout=0)),          # pixels-as-M generic kernel
    ('generic_swap', dict(strip=0, flat=0)),                      # weights-as-M generic kernel where 64 <= Cout <= 128
    ('flat', dict(strip=0, flat=2)),                              # flat halo-tile kernel wherever the shape is eligible
    ('strip_nofold', dict(fold=0)),                               # strip kernel, plain / swapped issue
    ('strip_plain', dict(fold=0, swap_min_cout=0)),               # strip kernel, pixels-as-M, 9 taps issued separately
    ('strip_no_nsplit', dict(nsplit=0)),
    ('strip_nsplit_two_launches', dict(nsplit=2)),                # default 1 = one launch of two-CTA clusters (TMA multicast)
    ('generic_tma_store', dict(strip=0, flat=0, swap_min_cout=0, tma_store=2)),   # generic kernel, outputs through TMA stores
    ('no_tma_store', dict(tma_store=0)),
    ('strip_pair', dict(pair=1)),                                 # folded strip loop on CTA-pair (cta_group::2) MMAs
    ('strip_single', dict(pair=0)),
]
WGRAD_VARIANTS = [('default', {}), ('generic', dict(wgrad_strip=0))]

CONV_CASES = [
    # N, H, W, C0, C1, Cout
    (1, 16, 16, 32, 0, 32),
    (2, 8, 24, 64, 0, 64),
    (1, 16, 16, 32, 32, 32),
    (2, 8, 8, 128, 128, 128),
    (3, 4, 4, 256, 0, 512),
    (1, 32, 32, 64, 64, 64),
    (1, 2, 2, 512, 0, 512),
    # wide rows (W % 128 == 0): the halo-strip kernel in bf16 mode
    (1, 8, 128, 32, 0, 32),
    (2, 5, 256, 64, 0, 64),
    (1, 20, 128, 32, 32, 32),
    (1, 1, 128, 32, 0, 64),
    (3, 37, 128, 64, 0, 32),
    (1, 9, 512, 32, 32, 32),
    (2, 11, 64, 32, 0, 64),
    (4, 128, 128, 32, 32, 32),
    (2, 6, 128, 64, 64, 64),      # weights too large for one strip launch: output channels split over a CTA pair / two launches
    (3, 38, 256, 64, 64, 64),
    (1, 4, 256, 64, 64, 64),
    # 64-channel sources on 64-pixel rows: strip wgrad over two / three / four 32-channel blocks
    (1, 16, 64, 64, 0, 64),
    (2, 8, 64, 64, 64, 64),
    (1, 8, 128, 64, 32, 32),
    # CTA-pair strip kernel: column pairs inside a row / across images, strips longer than the accumulator ring
    # (wrapping spans), every channel combination it takes
    (2, 8, 128, 32, 0, 32),
    (1, 6, 256, 32, 0, 64),
    (2, 44, 256, 64, 0, 32),
    (1, 40, 512, 64, 0, 64),
    (2, 36, 128, 32, 32, 64),
    # enough 256-pixel tiles for the swapped (weights-as-A) orientation of the generic kernel
    (8, 64, 64, 64, 0, 128),
    (5, 48, 80, 64, 64, 64),
    # the padded networks (nb_filters_base 48 / 64): more than 512 output channels (slices of 512 through the generic
    # kernel, with offsets into weights, scale, shift and output), concat inputs of 1536 and 768 channels
    (2, 4, 4, 512, 0, 768),
    (1, 4, 6, 512, 0, 1024),
    (2, 2, 2, 1024, 0, 1024),
    (1, 8, 8, 1024, 512, 512),
    (2, 8, 8, 512, 256, 256),
    # tiled inference: level widths of a 640 and a 192 tile at batch 8 (no W % 128 strip rows below 640)
    (8, 4, 640, 32, 0, 32),
    (8, 4, 320, 64, 0, 64),
    (8, 4, 160, 128, 128, 128),
    (8, 4, 80, 256, 0, 256),
    (8, 4, 192, 64, 0, 64),
    (8, 4, 96, 128, 0, 128),
    (3, 6, 640, 64, 64, 64),          # odd N
]


@pytest.mark.parametrize('precision', ['fp32', 'bf16', 'fp16'])
@pytest.mark.parametrize('case', CONV_CASES)
def test_conv3x3_fwd_dgrad_wgrad(cuda, precision, case):
    from deepcalcium.engine import ops
    N, H, W, C0, C1, Cout = case
    dt = DT[precision]
    rng = np.random.default_rng(hash(case) % 2**31)
    Cin = C0 + C1
    x = q(rng.standard_normal((N, H, W, Cin)), precision)
    w = q(rng.standard_normal((3, 3, Cin, Cout)) * np.sqrt(2. / (9 * Cin)), precision)
    scale = rng.uniform(0.5, 1.5, Cout).astype(np.float32)
    shift = rng.standard_normal(Cout).astype(np.float32)
    xt = nhwc_to_nchw(x).requires_grad_(True)
    wt = torch.tensor(w, requires_grad=True)
    conv = F.conv2d(xt, wt.permute(3, 2, 0, 1), padding=1)
    ref = torch.relu(conv * torch.tensor(scale, dtype=torch.float64)[None, :, None, None]
                     + torch.tensor(shift, dtype=torch.float64)[None, :, None, None])
    # the same contraction on absolute values: B of the rounding bound, forward / dgrad / wgrad
    xa = nhwc_to_nchw(np.abs(x)).requires_grad_(True)
    wa = torch.tensor(np.abs(w), requires_grad=True)
    conv_abs = F.conv2d(xa, wa.permute(3, 2, 0, 1), padding=1)
    from deepcalcium import _native as nat
    x0 = dev(x[..., :C0], dt)
    x1 = dev(x[..., C0:], dt) if C1 else None
    wm = dev(w)
    wf = torch.empty(9 * Cin * Cout, dtype=dt, device='cuda')
    wd = torch.empty(9 * Cin * Cout, dtype=dt, device='cuda')
    ops.prep_conv3x3_weights(wm, wf, wd, dt)
    dy = q(rng.standard_normal((N, H, W, Cout)), precision)
    conv.backward(nhwc_to_nchw(dy))
    conv_abs.backward(nhwc_to_nchw(np.abs(dy)))
    dyd = dev(dy, dt)
    seen = {}
    tc = precision != 'fp32'
    for vname, pol in (FWD_VARIANTS if tc else FWD_VARIANTS[:1]):
        with nat.policy(**pol):
            # forward (+ concat + epilogue)
            out = torch.empty(N, H, W, Cout, dtype=dt, device='cuda')
            ops.conv3x3_fwd(x0, x1, wf, out, dev(scale), dev(shift), True)
            kf = nat.last_kernel()
            if tc:
                got = out.cpu().permute(0, 3, 1, 2)
                r = assert_bound(got, conv, conv_abs, scale, shift, precision, (case, precision, vname, kf), c_acc=rb.c_acc_tc(9 * Cin))
            else:
                got = out.float().cpu().permute(0, 3, 1, 2).double()
                assert torch.max(torch.abs(got - ref)).item() < tol(precision, 1 + ref.abs().max().item()), (vname, kf)
            # plain conv (no epilogue): dgrad against autograd; gradients are fp32 in every mode
            dx = torch.empty(N, H, W, Cin, dtype=torch.float32, device='cuda')
            ops.conv3x3_dgrad(dyd, wd, dx)
            kd = nat.last_kernel()
            gx = dx.float().cpu().permute(0, 3, 1, 2).double()
            if tc:
                ra = assert_acc(gx, xt.grad, xa.grad, rb.c_acc_tc(9 * Cout), (case, precision, vname, kd))
                seen[vname] = (kf, kd, 'exact %.4f / %.4f sharp %.4f dgrad c %.2f' % (r['exact'], r['exact_nz'], r['sharp'], ra))
            else:
                assert torch.max(torch.abs(gx - xt.grad)).item() < tol(precision, 1 + xt.grad.abs().max().item()), (vname, kd)
    if tc:
        assert seen['generic'][0] == 'generic' and seen['generic_swap'][0] in ('generic', 'generic_swap')
        print('conv %s %s kernels: %s' % (case, precision, seen))
    if precision == 'fp16':           # fp16 is inference only: the library rejects fp16 gradients
        dW = torch.empty(3, 3, Cin, Cout, dtype=torch.float32, device='cuda')
        ws = torch.empty(max(16, ops.conv3x3_wgrad_workspace_bytes(torch.bfloat16, N, H, W, Cin, Cout)), dtype=torch.uint8, device='cuda')
        with pytest.raises(nat.DcbError):
            ops.conv3x3_wgrad(x0, x1, dyd, dW, ws)
        return
    for vname, pol in (WGRAD_VARIANTS if tc else WGRAD_VARIANTS[:1]):
        with nat.policy(**pol):
            dW = torch.empty(3, 3, Cin, Cout, dtype=torch.float32, device='cuda')
            ws = torch.empty(max(16, ops.conv3x3_wgrad_workspace_bytes(dt, N, H, W, Cin, Cout)), dtype=torch.uint8, device='cuda')
            ops.conv3x3_wgrad(x0, x1, dyd, dW, ws)
            gw = dW.cpu().double()
            if tc:
                assert_acc(gw, wt.grad, wa.grad, rb.C_ACC_WGRAD, (case, vname, nat.last_kernel()))
            else:
                assert torch.max(torch.abs(gw - wt.grad)).item() < tol(precision, 1 + wt.grad.abs().max().item()), (vname, nat.last_kernel())


def test_policy_roundtrip_and_kernel_names(cuda):
    """dcb_set_policy / dcb_get_policy / dcb_reset_policy and dcb_last_kernel: the variant actually launched is
    observable, so a test can tell which kernel it has verified."""
    from deepcalcium import _native as nat
    from deepcalcium.engine import ops
    nat.reset_policy()
    assert nat.get_policy('flat') == 1 and nat.get_policy('swap_min_cout') == 64
    with nat.policy(flat=2, strip=0):
        assert nat.get_policy('flat') == 2 and nat.get_policy('strip') == 0
    assert nat.get_policy('flat') == 1 and nat.get_policy('strip') == 1
    dt = torch.bfloat16

    def run(N, H, W, Cin, Cout):
        x = torch.zeros(N, H, W, Cin, dtype=dt, device='cuda')
        wf = torch.zeros(9 * Cin * Cout, dtype=dt, device='cuda')
        out = torch.empty(N, H, W, Cout, dtype=dt, device='cuda')
        ops.conv3x3_fwd(x, None, wf, out, None, None, False)
        return nat.last_kernel()
    assert run(1, 8, 128, 32, 32) == 'strip_fold'
    with nat.policy(fold=0):
        assert run(1, 4, 256, 64, 64) == 'strip_swap'
    with nat.policy(fold=0, swap_min_cout=0):
        assert run(1, 8, 128, 32, 32) == 'strip'
    with nat.policy(strip=0):
        assert run(1, 8, 128, 32, 32) == 'generic'
    with nat.policy(flat=2):
        assert run(2, 32, 32, 64, 64) == 'flat'
    assert run(2, 32, 32, 64, 64) in ('generic', 'generic_swap')          # too few work items for the flat kernel


CONVT_CASES = [
    # N, h, w, Cin, Cout
    (1, 8, 8, 64, 32), (2, 4, 4, 512, 256), (1, 16, 16, 128, 64), (3, 2, 2, 256, 128), (4, 64, 64, 128, 64), (8, 64, 64, 64, 32),
    (2, 4, 4, 1024, 512),          # up3 of nb_filters_base 64
    (8, 10, 10, 256, 128),         # a 640 tile's 80^2 level
]


@pytest.mark.parametrize('precision', ['fp32', 'bf16', 'fp16'])
@pytest.mark.parametrize('case', CONVT_CASES)
def test_convT2x2_fwd_dgrad_wgrad(cuda, precision, case):
    from deepcalcium.engine import ops
    N, h, w_, Cin, Cout = case
    dt = DT[precision]
    rng = np.random.default_rng(hash(case) % 2**31)
    x = q(rng.standard_normal((N, h, w_, Cin)), precision)
    k = q(rng.standard_normal((2, 2, Cout, Cin)) * np.sqrt(2. / (4 * Cout)), precision)
    bias = rng.standard_normal(Cout).astype(np.float32)
    xt = nhwc_to_nchw(x).requires_grad_(True)
    kt = torch.tensor(k, requires_grad=True)
    ref = F.conv_transpose2d(xt, kt.permute(3, 2, 0, 1), torch.tensor(bias, dtype=torch.float64), stride=2)
    xa = nhwc_to_nchw(np.abs(x)).requires_grad_(True)
    ka = torch.tensor(np.abs(k), requires_grad=True)
    ref_abs = F.conv_transpose2d(xa, ka.permute(3, 2, 0, 1), stride=2)
    tc = precision != 'fp32'
    wf = torch.empty(4 * Cin * Cout, dtype=dt, device='cuda')
    wd = torch.empty(4 * Cin * Cout, dtype=dt, device='cuda')
    ops.prep_convT2x2_weights(dev(k), wf, wd, dt)
    from deepcalcium import _native as nat
    for tma_store in (1, 0):        # epilogue through TMA stores (default) / plain 32-byte stores
        with nat.policy(tma_store=tma_store):
            out = torch.zeros(N, 2 * h, 2 * w_, Cout, dtype=dt, device='cuda')
            ops.convT2x2_fwd(dev(x, dt), wf, out, None, dev(bias), False)
            if tc:        # bias as the epilogue shift with scale 1: y = A + bias, no ReLU
                assert_bound(out.cpu().permute(0, 3, 1, 2), ref - torch.tensor(bias, dtype=torch.float64)[None, :, None, None],
                             ref_abs, np.ones(Cout), bias, precision, (case, precision, tma_store), c_acc=rb.c_acc_tc(Cin), relu=False)
            else:
                got = out.float().cpu().permute(0, 3, 1, 2).double()
                assert torch.max(torch.abs(got - ref)).item() < tol(precision, 1 + ref.abs().max().item()), tma_store
    dy = q(rng.standard_normal((N, 2 * h, 2 * w_, Cout)), precision)
    ref.backward(nhwc_to_nchw(dy))
    ref_abs.backward(nhwc_to_nchw(np.abs(dy)))
    dx = torch.empty(N, h, w_, Cin, dtype=torch.float32, device='cuda')
    ops.convT2x2_dgrad(dev(dy, dt), wd, dx)
    if tc:
        assert_acc(dx.cpu().permute(0, 3, 1, 2).double(), xt.grad, xa.grad, rb.c_acc_tc(4 * Cout), (case, precision, 'dgrad'))
    else:
        assert torch.max(torch.abs(dx.float().cpu().permute(0, 3, 1, 2).double() - xt.grad)).item() < \
            tol(precision, 1 + xt.grad.abs().max().item())
    dW = torch.empty(2, 2, Cout, Cin, dtype=torch.float32, device='cuda')
    ws = torch.empty(max(16, ops.convT2x2_wgrad_workspace_bytes(torch.bfloat16 if tc else dt, N, h, w_, Cin, Cout)),
                     dtype=torch.uint8, device='cuda')
    if precision == 'fp16':           # inference only: no fp16 gradients
        with pytest.raises(nat.DcbError):
            ops.convT2x2_wgrad(dev(x, dt), dev(dy, dt), dW, ws)
        return
    ops.convT2x2_wgrad(dev(x, dt), dev(dy, dt), dW, ws)
    if tc:
        assert_acc(dW.cpu().double(), kt.grad, ka.grad, rb.C_ACC_WGRAD, (case, precision, 'wgrad'))
    else:
        assert torch.max(torch.abs(dW.cpu().double() - kt.grad)).item() < tol(precision, 1 + kt.grad.abs().max().item())


FUSED_SHAPES = [
    # N, H, W, Cin, Cout
    (2, 16, 128, 32, 32), (1, 6, 256, 64, 64), (1, 8, 24, 32, 32), (2, 40, 256, 32, 32), (1, 44, 512, 64, 32),
    (2, 8, 512, 64, 64), (8, 4, 640, 64, 64),        # full-resolution 64 -> 64 (nfb 64)
    # pooled epilogue of the generic kernel: pixels-as-M tiles (several tile shapes, an N tile narrower than Cout),
    # weights-as-M tiles of 128x2 and 64x4 pixels
    (2, 32, 32, 128, 128), (3, 8, 8, 256, 256), (8, 64, 64, 128, 256),
    (8, 128, 128, 64, 128), (16, 64, 64, 64, 128), (1, 16, 128, 64, 128),
]


@pytest.mark.parametrize('precision', ['fp32', 'bf16', 'fp16'])
@pytest.mark.parametrize('shape', FUSED_SHAPES)
def test_conv3x3_fused_pool_and_head_equal_the_unfused_composition(cuda, precision, shape):
    """dcb_conv3x3_fwd_fused (max-pool / softmax head folded into the conv epilogue) must reproduce the separate
    kernels - including shapes where the library falls back to the unfused composition.  fp32: exactly.  bf16: the
    fused and the unfused launch may pick different tensor-core schedules (pixel-major, weight-major or row-folded
    accumulation), i.e. different fp32 summation orders, so a few outputs may differ by one bf16 rounding step."""
    from deepcalcium.engine import ops
    N, H, W, Cin, Cout = shape
    dt = DT[precision]
    rng = np.random.default_rng(5)
    x = dev(rng.standard_normal((N, H, W, Cin)), dt)
    w = dev(rng.standard_normal((3, 3, Cin, Cout)) * np.sqrt(2. / (9 * Cin)))
    wf = torch.empty(9 * Cin * Cout, dtype=dt, device='cuda')
    ops.prep_conv3x3_weights(w, wf, None, dt)
    scale = dev(rng.uniform(0.5, 1.5, Cout)); shift = dev(rng.standard_normal(Cout))
    hk = dev(rng.standard_normal((Cout, 2)) * 0.3); hb = dev(np.array([0.1, -0.2]))
    y = torch.empty(N, H, W, Cout, dtype=dt, device='cuda')
    ops.conv3x3_fwd(x, None, wf, y, scale, shift, True)
    pool = torch.empty(N, H // 2, W // 2, Cout, dtype=dt, device='cuda')
    ops.maxpool2x2(y, pool)
    logit = torch.empty(N, H, W, device='cuda'); prob = torch.empty(N, H, W, device='cuda')
    ops.head_fwd(y, hk, hb, logit, prob)
    from deepcalcium import _native as nat
    for pair in (1, 0):          # CTA-pair / single-CTA strip kernel (where the shape takes the strip kernel at all)
        with nat.policy(pair=pair):
            _check_fused(ops, nat, precision, shape, x, wf, scale, shift, hk, hb, y, pool, logit, prob)


OVERFLOW_VARIANTS = [('plain', {}, False), ('generic', dict(strip=0, flat=0, swap_min_cout=0), False),
                     ('generic_swap', dict(strip=0, flat=0), False),
                     ('generic_tma_store', dict(strip=0, flat=0, swap_min_cout=0, tma_store=2), False),
                     ('strip_pool', {}, True), ('generic_pool', dict(strip=0, flat=0), True)]


@pytest.mark.parametrize('variant', OVERFLOW_VARIANTS, ids=[v[0] for v in OVERFLOW_VARIANTS])
def test_fp16_outputs_past_65504_are_stored_as_inf(cuda, variant):
    """fp16 range: a scale that pushes outputs past the largest fp16 value.  Every stored value is RN16 of the result -
    +inf from 65520 up, 0 for the negative ones after ReLU - in the plain, TMA-store and pooled epilogues, and no other bit
    pattern (NaN, 65504, bf16 bits) appears.  This characterises the kernels; nothing clamps on purpose."""
    from deepcalcium import _native as nat
    from deepcalcium.engine import ops
    name, pol, pooled = variant
    N, H, W, Cin, Cout = 2, 8, 128, 64, 64
    dt = torch.float16
    rng = np.random.default_rng(65504)
    x = q(rng.standard_normal((N, H, W, Cin)), 'fp16')
    w = q(rng.standard_normal((3, 3, Cin, Cout)) * np.sqrt(2. / (9 * Cin)), 'fp16')
    scale = np.where(np.arange(Cout) % 2 == 0, 6e4, 0.7).astype(np.float32)      # even channels overflow where A > ~1.1
    shift = rng.standard_normal(Cout).astype(np.float32)
    xt, wt = nhwc_to_nchw(x), torch.tensor(w).permute(3, 2, 0, 1)
    A = F.conv2d(xt, wt, padding=1)
    B = F.conv2d(xt.abs(), wt.abs(), padding=1)
    wf = torch.empty(9 * Cin * Cout, dtype=dt, device='cuda')
    ops.prep_conv3x3_weights(dev(w), wf, None, dt)
    out = torch.empty(N, H, W, Cout, dtype=dt, device='cuda')
    pool = torch.empty(N, H // 2, W // 2, Cout, dtype=dt, device='cuda')
    with nat.policy(**pol):
        if pooled:
            ops.conv3x3_fwd_fused(dev(x, dt), None, wf, out, dev(scale), dev(shift), True, pool_out=pool)
        else:
            ops.conv3x3_fwd(dev(x, dt), None, wf, out, dev(scale), dev(shift), True)
        kern = nat.last_kernel()
    got = out.cpu().permute(0, 3, 1, 2)
    assert not bool(torch.isnan(got).any()) and not bool((got == -np.inf).any()), kern
    n_inf = int(torch.isinf(got).sum())
    assert n_inf > 1000, (kern, n_inf)
    # the bound admits exactly +inf where RN16(v - d) is +inf and only finite values where RN16(v + d) is finite
    r = assert_bound(got, A, B, scale, shift, 'fp16', (name, kern), c_acc=rb.c_acc_tc(9 * Cin))
    if pooled:                        # the pooled copy: bit for bit the 2x2 max of what was stored (either zero of a +-0 tie)
        want = F.max_pool2d(out.permute(0, 3, 1, 2).float(), 2).permute(0, 2, 3, 1).to(dt).contiguous()
        assert bool(((pool.view(torch.int16) == want.view(torch.int16)) | ((pool == 0) & (want == 0))).all()), kern
    print('fp16 overflow %s -> %s: %d inf, exact %.5f' % (name, kern, n_inf, r['exact']))


def _check_fused(ops, nat, precision, shape, x, wf, scale, shift, hk, hb, y, pool, logit, prob):
    y2 = torch.empty_like(y); pool2 = torch.empty_like(pool)
    ops.conv3x3_fwd_fused(x, None, wf, y2, scale, shift, True, pool_out=pool2)
    print('fused pool %s %s -> %s' % (precision, shape, nat.last_kernel() if precision != 'fp32' else 'fp32 composition'))
    def same(a, b):
        if precision == 'fp32':
            return torch.equal(a, b)
        a, b = a.float(), b.float()
        return bool(((a - b).abs() <= 2.0 ** -7 * b.abs().clamp(min=1.0)).all()) and float((a != b).float().mean()) < 5e-3
    assert same(y2, y) and same(pool2, pool)
    y3 = torch.full_like(y, 7.0); logit3 = torch.empty_like(logit); prob3 = torch.empty_like(prob)
    ops.conv3x3_fwd_fused(x, None, wf, y3, scale, shift, True, head_kernel=hk, head_bias=hb, logit=logit3, prob=prob3,
                          need_y=False)
    # bf16: with need_y=False the fused kernel never rounds the activation to bf16 (it is not stored), the unfused
    # composition reads the rounded tensor: 32 terms x 2^-9 relative rounding each
    atol = 1e-5 if precision == 'fp32' else 5e-2
    assert torch.allclose(logit3, logit, atol=atol, rtol=1e-5) and torch.allclose(prob3, prob, atol=atol / 4)


@pytest.mark.parametrize('precision', ['fp32', 'bf16', 'fp16'])
@pytest.mark.parametrize('shape', [(2, 24, 40, 32), (3, 7, 33, 32), (1, 5, 130, 32), (4, 128, 128, 32), (2, 9, 21, 16), (1, 16, 16, 64),
                                   (8, 8, 640, 64)])
def test_conv3x3_first_layer_c1(cuda, precision, shape):
    """Cin = 1 layer (enc0a): CUDA-core forward; weight gradient = row-staged kernel for Cout == 32 (odd widths, one-row
    CTAs, more CTAs than rows), pixel-range kernel otherwise."""
    from deepcalcium.engine import ops
    dt = DT[precision]
    rng = np.random.default_rng(11)
    N, H, W, Cout = shape
    x = rng.standard_normal((N, H, W)).astype(np.float32)
    w = (rng.standard_normal((3, 3, 1, Cout)) * 0.5).astype(np.float32)
    b = rng.standard_normal(Cout).astype(np.float32)
    xt = torch.tensor(x, dtype=torch.float64)[:, None]
    wt = torch.tensor(w, dtype=torch.float64, requires_grad=True)
    ref = F.conv2d(xt, wt.permute(3, 2, 0, 1), torch.tensor(b, dtype=torch.float64), padding=1)
    out = torch.empty(N, H, W, Cout, dtype=dt, device='cuda')
    ops.conv3x3_c1_fwd(dev(x), dev(w), out, None, dev(b), False)
    if precision != 'fp32':
        A = F.conv2d(xt, wt.detach().permute(3, 2, 0, 1), padding=1)
        B = F.conv2d(xt.abs(), wt.detach().abs().permute(3, 2, 0, 1), padding=1)
        assert_bound(out.cpu().permute(0, 3, 1, 2), A, B, np.ones(Cout), b, precision, (shape, precision), c_acc=rb.C_ACC_C1,
                     relu=False)
    assert torch.max(torch.abs(out.float().cpu().permute(0, 3, 1, 2).double() - ref)).item() < tol(precision, 4)
    if precision == 'fp16':           # inference only: the weight gradient is not built for fp16
        return
    dy = q(rng.standard_normal((N, H, W, Cout)), precision)
    ref.backward(nhwc_to_nchw(dy))
    dW = torch.empty(3, 3, 1, Cout, dtype=torch.float32, device='cuda')
    ws = torch.empty(ops.conv3x3_c1_wgrad_workspace_bytes(Cout), dtype=torch.uint8, device='cuda')
    ops.conv3x3_c1_wgrad(dev(x), dev(dy, dt), dW, ws)
    assert torch.max(torch.abs(dW.cpu().double() - wt.grad)).item() < 2e-3 * (1 + wt.grad.abs().max().item())


@pytest.mark.parametrize('precision', ['fp32', 'bf16'])
@pytest.mark.parametrize('C', [32, 128, 512])
def test_batchnorm_train_forward_backward(cuda, precision, C):
    """stats -> finalize -> apply and the two backward kernels against autograd of the Keras formula
    (eps 1e-3, biased variance, momentum update), including the strided dy view of a concat gradient."""
    from deepcalcium.engine import ops
    dt = DT[precision]
    rng = np.random.default_rng(C)
    M = 1000
    x = q(rng.standard_normal((M, C)) * 2 + 0.5, precision)
    gamma = rng.uniform(0.5, 1.5, C).astype(np.float32); beta = (0.1 * rng.standard_normal(C)).astype(np.float32)
    mm = rng.standard_normal(C).astype(np.float32); mv = rng.uniform(0.5, 1.5, C).astype(np.float32)
    xt = torch.tensor(x, requires_grad=True)
    gt = torch.tensor(gamma, dtype=torch.float64, requires_grad=True)
    bt = torch.tensor(beta, dtype=torch.float64, requires_grad=True)
    mean = xt.mean(0); var = ((xt - mean) ** 2).mean(0)
    y = torch.relu((xt - mean) * torch.rsqrt(var + 1e-3) * gt + bt)
    xd = dev(x, dt).view(1, 1, M, C)
    sums = torch.zeros(4 * C, dtype=torch.float64, device='cuda')
    f = lambda: torch.empty(C, device='cuda')
    scale, shift, mean_d, rstd_d = f(), f(), f(), f()
    mmd, mvd = dev(mm), dev(mv)
    ops.bn_stats(xd, sums[:2 * C])
    ops.bn_finalize(sums[:2 * C], M, dev(gamma), dev(beta), 0.5, mmd, mvd, scale, shift, mean_d, rstd_d)
    yd = torch.empty_like(xd)
    ops.bn_apply(xd, scale, shift, yd, True)
    assert torch.max(torch.abs(yd.float().cpu().view(M, C).double() - y.detach())).item() < tol(precision, 4)
    assert np.allclose(mean_d.cpu().numpy(), mean.detach().numpy(), atol=1e-5)
    assert np.allclose(mmd.cpu().numpy(), mm * 0.5 + mean.detach().numpy() * 0.5, atol=1e-5)
    assert np.allclose(mvd.cpu().numpy(), mv * 0.5 + var.detach().numpy() * 0.5, atol=1e-4)
    # backward with dy living at channel offset C/2.. of a wider tensor (row stride 2C)
    dy_wide = q(rng.standard_normal((M, 2 * C)), precision)
    off = C // 2 if (C // 2) % 4 == 0 else 0
    dy = dy_wide[:, off:off + C]
    y.backward(torch.tensor(dy))
    draw = torch.empty_like(xd)
    dg, db = f(), f()
    dyd = dev(dy_wide)                                   # gradient tensors are fp32
    ops.bn_bwd_reduce(dyd, 2 * C, off, xd, scale, shift, mean_d, rstd_d, sums[2 * C:])
    ops.bn_bwd_apply(dyd, 2 * C, off, xd, scale, shift, mean_d, rstd_d, sums[2 * C:], draw, dg, db)
    t = tol(precision, 4)
    assert torch.max(torch.abs(draw.float().cpu().view(M, C).double() - xt.grad)).item() < t
    assert np.allclose(dg.cpu().numpy(), gt.grad.numpy(), atol=t * 30, rtol=1e-2 if precision == 'bf16' else 1e-4)
    assert np.allclose(db.cpu().numpy(), bt.grad.numpy(), atol=t * 30, rtol=1e-2 if precision == 'bf16' else 1e-4)


@pytest.mark.parametrize('precision', ['fp32', 'bf16'])
@pytest.mark.parametrize('slab', [2, 1, 0])
@pytest.mark.parametrize('shape', [(2, 16, 24, 32), (4, 32, 32, 64), (3, 8, 8, 512), (32, 128, 128, 32), (1, 2, 2, 128),
                                   # the levels of a 32 x 128^2 training step that run as channel-slab cluster kernels
                                   (32, 64, 64, 64), (32, 32, 32, 128), (32, 16, 16, 256), (32, 8, 8, 512), (5, 12, 20, 128)])
def test_single_launch_batchnorm_equals_the_separate_passes(cuda, precision, shape, slab):
    """dcb_bn_train_fwd / dcb_bn_train_bwd (one launch each: grid barriers with fixed-order cross-CTA sums, or - slab=2:
    wherever the shape is eligible, slab=1: small tensors only, the default - channel-slab clusters reducing through distributed shared memory; optional fused 2x2
    max-pool) against the four separate kernels they replace (each of which is checked against autograd above);
    and bit-for-bit run-to-run reproducibility, which the fp64-atomic version could not promise."""
    from deepcalcium import _native as nat
    with nat.policy(bn_slab=slab):
        _check_single_launch_batchnorm(precision, shape)


def _check_single_launch_batchnorm(precision, shape):
    from deepcalcium.engine import ops
    dt = DT[precision]
    N, H, W, C = shape
    M = N * H * W
    rng = np.random.default_rng(C + M)
    x = dev(rng.standard_normal((N, H, W, C)) * 2 + 0.5, dt)
    gamma = dev(rng.uniform(0.5, 1.5, C)); beta = dev(0.1 * rng.standard_normal(C))
    mm0 = rng.standard_normal(C).astype(np.float32); mv0 = rng.uniform(0.5, 1.5, C).astype(np.float32)
    f = lambda: torch.empty(C, device='cuda')
    ws = torch.zeros(ops.bn_train_workspace_bytes(C), dtype=torch.uint8, device='cuda')
    seed_dev = torch.tensor([4242], dtype=torch.int64, device='cuda')
    p_drop = 0.25
    # ---- separate passes
    sums = torch.zeros(4 * C, dtype=torch.float64, device='cuda')
    sc0, sh0, mu0, rs0 = f(), f(), f(), f()
    mm, mv = dev(mm0), dev(mv0)
    y0 = torch.empty_like(x); pool0 = torch.empty(N, H // 2, W // 2, C, dtype=dt, device='cuda')
    ops.bn_stats(x, sums[:2 * C])
    ops.bn_finalize_apply(x, sums[:2 * C], M, gamma, beta, 0.99, mm, mv, sc0, sh0, mu0, rs0, y0, True, p_drop, 7, seed_dev, 5)
    ops.maxpool2x2(y0, pool0)
    # ---- single launch, twice (determinism)
    outs = []
    for rep in range(2):
        sc, sh, mu, rs = f(), f(), f(), f()
        mm1, mv1 = dev(mm0), dev(mv0)
        y = torch.empty_like(x); pool = torch.empty_like(pool0)
        sync = torch.zeros(4, dtype=torch.int32, device='cuda')
        ops.bn_train_fwd(x, gamma, beta, 0.99, mm1, mv1, sc, sh, mu, rs, y, ws, sync, True, p_drop, 7, seed_dev, 5, pool_out=pool)
        outs.append((y, pool, sc, sh, mu, rs, mm1, mv1))
    for a, b in zip(*outs):
        assert torch.equal(a, b)
    y, pool, sc, sh, mu, rs, mm1, mv1 = outs[0]
    for a, b in ((sc, sc0), (sh, sh0), (mu, mu0), (rs, rs0), (mm1, mm), (mv1, mv)):
        assert torch.allclose(a, b, rtol=2e-6, atol=2e-6)
    step = 2.0 ** -7 if precision == 'bf16' else 1e-5
    assert float(((y.float() - y0.float()).abs() > step * y0.float().abs().clamp(min=1.0)).float().mean()) == 0.0
    # bit-level agreement with the separate passes: a scale that lands one fp32 ulp away (different summation tree) moves
    # every element of its channel by an ulp, which only shows in the fp32 mode
    if precision == 'bf16':
        assert float((y != y0).float().mean()) < 1e-3 and float((pool != pool0).float().mean()) < 1e-3
    pool_chk = torch.empty_like(pool0)
    ops.maxpool2x2(y, pool_chk)                                           # the fused pool is exactly the pool of what was stored
    assert torch.equal(pool, pool_chk)
    y_np = torch.empty_like(x)                                            # no pooling: same activations
    sync = torch.zeros(4, dtype=torch.int32, device='cuda')
    ops.bn_train_fwd(x, gamma, beta, 0.99, dev(mm0), dev(mv0), f(), f(), f(), f(), y_np, ws, sync, True, p_drop, 7, seed_dev, 5)
    # (the pooled instantiation may run a different grid, i.e. another summation tree: an fp32 scale can move by an ulp)
    assert torch.equal(y_np, y) if precision == 'bf16' else torch.allclose(y_np, y, rtol=1e-5, atol=1e-5)
    # ---- backward: dy is a channel slice of a wider fp32 tensor
    dy_wide = dev(rng.standard_normal((M, 2 * C)))
    off = C // 2 if (C // 2) % 4 == 0 else 0
    draw0 = torch.empty_like(x); dg0, db0 = f(), f()
    ops.bn_bwd_reduce(dy_wide, 2 * C, off, x, sc0, sh0, mu0, rs0, sums[2 * C:], p_drop, 7, seed_dev, 5)
    ops.bn_bwd_apply(dy_wide, 2 * C, off, x, sc0, sh0, mu0, rs0, sums[2 * C:], draw0, dg0, db0, p_drop, 7, seed_dev, 5)
    res = []
    for rep in range(2):
        draw = torch.empty_like(x); dg, db = f(), f()
        sync = torch.zeros(4, dtype=torch.int32, device='cuda')
        ops.bn_train_bwd(dy_wide, 2 * C, off, x, sc0, sh0, mu0, rs0, draw, dg, db, ws, sync, p_drop, 7, seed_dev, 5)
        res.append((draw, dg, db))
    for a, b in zip(*res):
        assert torch.equal(a, b)
    draw, dg, db = res[0]
    scale_g = float(draw0.float().abs().max())
    assert float((draw.float() - draw0.float()).abs().max()) <= (2.0 ** -7 if precision == 'bf16' else 1e-5) * scale_g
    assert torch.allclose(dg, dg0, rtol=1e-5, atol=1e-4) and torch.allclose(db, db0, rtol=1e-5, atol=1e-4)
    # in place (draw aliases x), as the engine uses it
    x2 = x.clone(); sync = torch.zeros(4, dtype=torch.int32, device='cuda')
    ops.bn_train_bwd(dy_wide, 2 * C, off, x2, sc0, sh0, mu0, rs0, x2, f(), f(), ws, sync, p_drop, 7, seed_dev, 5)
    assert torch.equal(x2, draw)


@pytest.mark.parametrize('precision', ['fp32', 'bf16', 'fp16'])
def test_maxpool_forward_and_backward_routing(cuda, precision):
    from deepcalcium.engine import ops
    dt = DT[precision]
    rng = np.random.default_rng(3)
    N, H, W, C = 2, 8, 12, 32
    x = q(np.maximum(rng.standard_normal((N, H, W, C)), 0), precision)     # ReLU output: many tied zeros
    xt = nhwc_to_nchw(x).requires_grad_(True)
    ref = F.max_pool2d(xt, 2)
    xd = dev(x, dt)
    yd = torch.empty(N, H // 2, W // 2, C, dtype=dt, device='cuda')
    ops.maxpool2x2(xd, yd)
    assert torch.equal(yd.float().cpu().permute(0, 3, 1, 2).double(), ref.detach())
    if precision == 'fp16':           # inference only: forward
        return
    dp = q(rng.standard_normal((N, H // 2, W // 2, C)), precision)
    skip_wide = q(rng.standard_normal((N, H, W, 2 * C)), precision)
    ref.backward(nhwc_to_nchw(dp))
    out = torch.empty(N, H, W, C, dtype=torch.float32, device='cuda')
    ops.pool_bwd_add(dev(skip_wide), 2 * C, C, xd, yd, dev(dp), out)
    exp = xt.grad + nhwc_to_nchw(skip_wide[..., C:])
    # every pooled gradient lands on exactly one input pixel (torch also picks the first maximum)
    assert torch.max(torch.abs(out.float().cpu().permute(0, 3, 1, 2).double() - exp)).item() < tol(precision, 4)


@pytest.mark.parametrize('precision', ['fp32', 'bf16', 'fp16'])
@pytest.mark.parametrize('loss', ['dice_loss', 'binary_crossentropy', 'dicesq_loss', 'weighted_binary_crossentropy'])
def test_head_loss_metrics_and_gradient(cuda, precision, loss):
    from deepcalcium.engine import ops
    from deepcalcium import _native as nat
    dt = DT[precision]
    rng = np.random.default_rng(17)
    M, C = 3000, 32
    x = q(rng.standard_normal((M, C)), precision)
    w = (rng.standard_normal((C, 2)) * 0.3).astype(np.float32); b = np.array([0.1, -0.2], np.float32)
    yt = (rng.random(M) < 0.126).astype(np.uint8)
    xt = torch.tensor(x, requires_grad=True)
    wt = torch.tensor(w, dtype=torch.float64, requires_grad=True); bt = torch.tensor(b, dtype=torch.float64, requires_grad=True)
    p = torch.softmax(xt @ wt + bt, dim=1)[:, -1]
    L = ol.LOSSES[loss](torch.tensor(yt, dtype=torch.float64), p)
    L.backward()
    xd = dev(x, dt).view(1, 1, M, C)
    prob = torch.empty(M, device='cuda'); logit = torch.empty(M, device='cuda')
    ops.head_fwd(xd, dev(w), dev(b), logit, prob)
    assert np.allclose(prob.cpu().numpy(), p.detach().numpy(), atol=1e-5)
    if precision == 'fp16':           # inference only: head_fwd
        return
    sums = torch.zeros(8, dtype=torch.float64, device='cuda'); dwb = torch.zeros(2 * C + 2, dtype=torch.float64, device='cuda')
    ops.head_loss_fwd(xd, dev(w), dev(b), dev(yt, torch.uint8), prob, sums)
    dx = torch.empty(1, 1, M, C, device='cuda'); dw = torch.empty(2 * C + 2, device='cuda'); met = torch.empty(8, device='cuda')
    ops.head_loss_bwd(xd, dev(w), dev(yt, torch.uint8), prob, sums, nat.LOSS_IDS[loss], dx, dwb, dw, met)
    met = met.cpu().numpy()
    assert abs(met[0] - L.item()) < 2e-5 * max(1, abs(L.item()))
    om = ol.batch_metrics(yt, p.detach().numpy())
    for i, k in enumerate(['F1', 'prec', 'reca', 'dice', 'dicesq', 'posyt', 'posyp']):
        assert abs(met[1 + i] - om[k]) < 1e-4, k
    gscale = xt.grad.abs().max().item()
    assert torch.max(torch.abs(dx.float().cpu().view(M, C).double() - xt.grad)).item() < (1e-2 if precision == 'bf16' else 1e-4) * gscale + 1e-9
    assert np.allclose(dw[:2 * C].cpu().numpy().reshape(C, 2), wt.grad.numpy(), rtol=1e-3, atol=1e-5 * (1 + wt.grad.abs().max().item()))
    assert np.allclose(dw[2 * C:].cpu().numpy(), bt.grad.numpy(), rtol=1e-3, atol=1e-6)


def test_tta_batch_and_combine_match_the_reference_table(cuda):
    from deepcalcium.engine import ops
    from deepcalcium.utils.neurons import INVERTIBLE_2D_AUGMENTATIONS as TABLE
    rng = np.random.default_rng(4)
    S, hs, ws = 32, 27, 30
    s = rng.standard_normal((hs, ws)).astype(np.float32)
    padded = oracle.reflect_pad(s, S, S)[None]
    out = torch.empty(8, S, S, device='cuda')
    ops.tta_make_batch(dev(s), S, 0, 8, out)
    for k, (name, aug, inv) in enumerate(TABLE):
        assert np.array_equal(out[k].cpu().numpy(), aug(padded)[0]), name
    sub = torch.empty(3, S, S, device='cuda')
    ops.tta_make_batch(dev(s), S, 4, 3, sub)
    assert torch.equal(sub, out[4:7])
    probs = rng.random((8, S, S)).astype(np.float32)
    mp = np.zeros((hs, ws))
    for k, (name, aug, inv) in enumerate(TABLE):
        mp += inv(probs[k:k + 1])[0, :hs, :ws] / len(TABLE)
    act = torch.empty(hs, ws, dtype=torch.float64, device='cuda'); mask = torch.empty(hs, ws, dtype=torch.uint8, device='cuda')
    ops.tta_combine(dev(probs), S, hs, ws, 0.5, 8, act, mask)
    assert np.array_equal(act.cpu().numpy(), mp)                       # same fp32 /8 then fp64 adds, same order
    assert np.array_equal(mask.cpu().numpy(), (mp > 0.5).astype(np.uint8))
    ops.tta_combine(dev(probs), S, hs, ws, 0.5, 1, act, mask)
    assert np.array_equal(mask.cpu().numpy(), (probs[0, :hs, :ws] > 0.5).astype(np.uint8))


def test_keras_adam_kernel(cuda):
    from deepcalcium.engine import ops
    rng = np.random.default_rng(9)
    n = 10001
    p = rng.standard_normal(n); g = rng.standard_normal(n) * 1e-3
    m = np.zeros(n); v = np.zeros(n)
    pd, md, vd = dev(p), dev(m), dev(v)
    state = torch.zeros(2, dtype=torch.int64, device='cuda'); lr_t = torch.zeros(1, device='cuda')
    for it in range(3):
        gi = g * (it + 1)
        p, m, v = oracle.keras_adam_update(p, gi, m, v, it, lr=0.002)
        ops.step_advance(state, 0.002, 0.9, 0.999, lr_t)
        ops.adam_step(pd, dev(gi), md, vd, 0., lr_t)
    assert state[0].item() == 3
    assert np.allclose(pd.cpu().numpy(), p, atol=2e-6)
    assert np.allclose(vd.cpu().numpy(), v, rtol=1e-4, atol=1e-12)


@pytest.mark.parametrize('precision', ['fp32', 'bf16'])
def test_bn_finalize_apply_equals_the_two_separate_calls(cuda, precision):
    from deepcalcium.engine import ops
    dt = DT[precision]
    rng = np.random.default_rng(3)
    for M, C in ((700, 32), (96, 4), (64, 512)):
        x = dev(rng.standard_normal((M, C)) * 2 + 0.5, dt)
        gamma = dev(rng.uniform(0.5, 1.5, C)); beta = dev(rng.standard_normal(C))
        mm0 = rng.standard_normal(C).astype(np.float32); mv0 = rng.uniform(0.5, 1.5, C).astype(np.float32)
        sums = torch.zeros(2 * C, dtype=torch.float64, device='cuda')
        ops.bn_stats(x, sums)
        outs = []
        for fused in (False, True):
            mm, mv = dev(mm0), dev(mv0)
            sc, sh, mu, rs = (torch.empty(C, device='cuda') for _ in range(4))
            y = torch.empty_like(x)
            if fused:
                ops.bn_finalize_apply(x, sums, M, gamma, beta, 0.99, mm, mv, sc, sh, mu, rs, y, True, 0.25, 77, None, 5)
            else:
                ops.bn_finalize(sums, M, gamma, beta, 0.99, mm, mv, sc, sh, mu, rs)
                ops.bn_apply(x, sc, sh, y, True, 0.25, 77, None, 5)
            outs.append([t.clone() for t in (y, sc, sh, mu, rs, mm, mv)])
        for a, b in zip(*outs):
            assert torch.equal(a, b)


@pytest.mark.parametrize('precision', ['fp32', 'bf16', 'fp16'])
def test_prep_weights_batch_equals_per_layer_calls(cuda, precision):
    from deepcalcium.engine import ops
    dt = DT[precision]
    rng = np.random.default_rng(4)
    layers = [('conv', 32, 64), ('convT', 64, 32), ('conv', 1, 32), ('conv', 96, 32), ('conv', 1536, 512), ('convT', 1024, 512)]
    rows, ref, got = [], [], []
    for kind, cin, cout in layers:
        if kind == 'conv':
            w = dev(rng.standard_normal((3, 3, cin, cout)))
            n = 9 * cin * cout
        else:
            w = dev(rng.standard_normal((2, 2, cout, cin)))
            n = 4 * cin * cout
        wf, wd, wf2, wd2 = (torch.zeros(n, dtype=dt, device='cuda') for _ in range(4))
        (ops.prep_conv3x3_weights if kind == 'conv' else ops.prep_convT2x2_weights)(w, wf, wd, dt)
        rows.append([w.data_ptr(), wf2.data_ptr(), wd2.data_ptr(), cin | (cout << 32), 0 if kind == 'conv' else 1])
        ref += [wf, wd]; got += [wf2, wd2]; rows[-1].append(w)      # keep w alive
    tab = torch.tensor([r[:5] for r in rows], dtype=torch.int64, device='cuda')
    ops.prep_weights_batch(tab, len(rows), dt)
    for a, b in zip(ref, got):
        assert torch.equal(a.view(torch.int16) if dt != torch.float32 else a, b.view(torch.int16) if dt != torch.float32 else b)
    if dt != torch.float32:           # both are round-to-nearest of the fp32 master: [Cout][9][Cin] / [4][Cout][Cin]
        w0 = rows[0][5]
        assert torch.equal(ref[0].view(torch.int16), w0.permute(3, 0, 1, 2).reshape(-1).to(dt).view(torch.int16))
        w1 = rows[1][5]
        assert torch.equal(ref[2].view(torch.int16), w1.reshape(-1).to(dt).view(torch.int16))


STATS_CASES = [
    # kind, shape, policy          conv: (N, H, W, C0, C1, Cout)   convT: (N, h, w, Cin, Cout)   c1: (N, H, W, Cout)
    ('conv', (3, 4, 4, 256, 0, 512), {}),                   # generic kernel, two N tiles
    ('conv', (2, 8, 8, 128, 128, 128), {}),
    ('conv', (1, 32, 32, 64, 64, 64), {}),
    ('conv', (2, 8, 24, 64, 0, 64), {}),                    # ragged tiles: out-of-image lanes must not count
    ('conv', (1, 2, 2, 512, 0, 512), {}),
    ('conv', (5, 48, 80, 64, 64, 64), {}),
    ('conv', (32, 16, 16, 128, 0, 256), {}),
    ('conv', (1, 8, 128, 32, 0, 32), {}),                   # folded strip kernel
    ('conv', (4, 128, 128, 32, 32, 32), {}),
    ('conv', (2, 44, 256, 64, 0, 32), {}),
    ('conv', (1, 6, 256, 32, 0, 64), {}),
    ('conv', (3, 37, 128, 64, 0, 32), {}),                  # odd height: no folded strip -> statistics not available there
    ('conv', (8, 64, 64, 64, 0, 128), dict(flat=2)),        # flat halo-tile kernel
    ('conv', (4, 32, 32, 64, 64, 256), dict(flat=2)),       # ... two channel tiles
    ('conv', (2, 40, 64, 64, 0, 64), dict(flat=2)),
    ('convT', (1, 8, 8, 64, 32), {}),
    ('convT', (2, 4, 4, 512, 256), {}),
    ('convT', (1, 16, 16, 128, 64), {}),
    ('convT', (3, 2, 2, 256, 128), {}),
    ('convT', (4, 64, 64, 64, 32), {}),
    ('convT', (2, 5, 7, 64, 32), {}),
    ('c1', (4, 128, 128, 32), {}),
    ('c1', (3, 7, 33, 32), {}),
]


@pytest.mark.parametrize('case', STATS_CASES)
def test_conv_epilogue_batch_statistics(cuda, case):
    """dcb_conv*_fwd_stats (training forward, bf16): the output equals the plain call's and sums = per-channel sum / sum of
    squares of the STORED output (fp64 reference from the output itself); two runs give bit-identical sums (fixed-order fp32
    partials, integer cross-CTA totals)."""
    from deepcalcium import _native as nat
    from deepcalcium.engine import ops
    kind, shape, pol = case
    import zlib
    rng = np.random.default_rng(zlib.crc32(str(case).encode()))
    bf = torch.bfloat16
    with nat.policy(swap_min_cout=0, fused_bn=3, **pol):
        if kind == 'conv':
            N, H, W, C0, C1, Cout = shape
            x0 = dev(rng.standard_normal((N, H, W, C0)), bf)
            x1 = dev(rng.standard_normal((N, H, W, C1)), bf) if C1 else None
            wk = (rng.standard_normal((3, 3, C0 + C1, Cout)) * np.sqrt(2.0 / (9 * (C0 + C1)))).astype(np.float32)
            wf = torch.empty(9 * (C0 + C1) * Cout, dtype=bf, device='cuda')
            ops.prep_conv3x3_weights(dev(wk), wf, None, bf)
            bias = dev(0.3 * rng.standard_normal(Cout))
            ref = torch.empty(N, H, W, Cout, dtype=bf, device='cuda')
            run_ref = lambda: ops.conv3x3_fwd(x0, x1, wf, ref, None, bias, False)
            run = lambda out, sums: ops.conv3x3_fwd_stats(x0, x1, wf, out, sums, None, bias, False)
        elif kind == 'convT':
            N, h, w_, Cin, Cout = shape
            x0 = dev(rng.standard_normal((N, h, w_, Cin)), bf)
            wk = (rng.standard_normal((2, 2, Cout, Cin)) * np.sqrt(2.0 / (4 * Cin))).astype(np.float32)
            wf = torch.empty(4 * Cin * Cout, dtype=bf, device='cuda')
            ops.prep_convT2x2_weights(dev(wk), wf, None, bf)
            bias = dev(0.3 * rng.standard_normal(Cout))
            ref = torch.empty(N, 2 * h, 2 * w_, Cout, dtype=bf, device='cuda')
            run_ref = lambda: ops.convT2x2_fwd(x0, wf, ref, None, bias, False)
            run = lambda out, sums: ops.convT2x2_fwd_stats(x0, wf, out, sums, None, bias, False)
        else:
            N, H, W, Cout = shape
            x0 = dev(rng.standard_normal((N, H, W)))
            wk = dev((rng.standard_normal((3, 3, 1, Cout)) * 0.5).astype(np.float32))
            bias = dev(0.3 * rng.standard_normal(Cout))
            ref = torch.empty(N, H, W, Cout, dtype=bf, device='cuda')
            run_ref = lambda: ops.conv3x3_c1_fwd(x0, wk, ref, None, bias, False)
            run = lambda out, sums: ops.conv3x3_c1_fwd_stats(x0, wk, out, sums, None, bias, False)
        run_ref()
        results = []
        for rep in range(2):
            out = torch.zeros_like(ref)
            sums_q = torch.zeros(2 * Cout, dtype=torch.int64, device='cuda')
            done = run(out, sums_q)
            sums = sums_q.double() / 2 ** 20
            kern = nat.last_kernel()
            torch.cuda.synchronize()
            # same accumulation, possibly a different tile order: identical up to bf16 rounding of equal fp32 values
            assert torch.max(torch.abs(out.float() - ref.float())).item() <= 2e-2 * max(1.0, ref.float().abs().max().item())
            if done:
                o = out.double().reshape(-1, Cout)
                want = torch.cat([o.sum(0), (o * o).sum(0)])
                err = (sums - want).abs() / (want.abs() + 1e-3 * o.shape[0])
                assert err.max().item() < 2e-5, (kern, err.max().item())
            results.append((done, sums_q.clone()))
        assert results[0][0] == results[1][0]
        if results[0][0]:
            assert torch.equal(results[0][1], results[1][1])
        print('%s %s -> %s, statistics %s' % (kind, shape, kern, 'in the epilogue' if results[0][0] else 'not available'))
        if kind == 'conv' and shape[2] % 128 == 0 and shape[1] % 2 == 0 and Cout <= 64:
            assert results[0][0] and kern == 'strip_fold_stats'
        if pol.get('flat') == 2:
            assert results[0][0] and kern == 'flat_stats'
        if kind == 'convT':
            assert results[0][0] and kern == 'generic_stats'


@pytest.mark.parametrize('shape', [(2, 16, 24, 32), (4, 32, 32, 64), (3, 8, 8, 512), (8, 128, 128, 32)])
@pytest.mark.parametrize('pool', [False, True])
def test_batchnorm_from_known_sums_equals_the_single_launch_kernel(cuda, shape, pool):
    """dcb_bn_train_fwd_sums (one pass from the batch sums a conv epilogue took) against dcb_bn_train_fwd on the same
    tensor: activation, pooled copy, coefficients and moving statistics."""
    from deepcalcium.engine import ops
    N, H, W, C = shape
    rng = np.random.default_rng(C + H)
    bf = torch.bfloat16
    x = dev(rng.standard_normal((N, H, W, C)) * 1.7 + 0.4, bf)
    gamma, beta = dev(rng.uniform(0.5, 1.5, C)), dev(0.1 * rng.standard_normal(C))
    f = lambda: torch.empty(C, device='cuda')
    outs = []
    for mode in ('fused', 'sums'):
        mm, mv = dev(np.linspace(-1, 1, C)), dev(np.linspace(0.5, 1.5, C))
        scale, shift, mean, rstd = f(), f(), f(), f()
        y = torch.empty_like(x)
        p = torch.empty(N, H // 2, W // 2, C, dtype=bf, device='cuda') if pool else None
        if mode == 'fused':
            wsb = torch.zeros(ops.bn_train_workspace_bytes(C), dtype=torch.uint8, device='cuda')
            sync = torch.zeros(4, dtype=torch.int32, device='cuda')
            ops.bn_train_fwd(x, gamma, beta, 0.99, mm, mv, scale, shift, mean, rstd, y, wsb, sync, True, 0.25, 11, None, 3, pool_out=p)
        else:
            o = x.double().reshape(-1, C)
            sums = torch.round(torch.cat([o.sum(0), (o * o).sum(0)]) * 2 ** 20).to(torch.int64).contiguous()
            ops.bn_train_fwd_sums(x, sums, gamma, beta, 0.99, mm, mv, scale, shift, mean, rstd, y, True, 0.25, 11, None, 3, pool_out=p)
        torch.cuda.synchronize()
        outs.append((y, p, scale, shift, mean, rstd, mm, mv))
    a, b = outs
    for i in (2, 3, 4, 5, 6, 7):
        assert torch.allclose(a[i], b[i], rtol=1e-5, atol=1e-6), i
    # coefficients agree to fp32 rounding, so the 16-bit activations agree except for rare one-ulp flips
    assert (a[0].float() - b[0].float()).abs().max().item() <= 4e-2
    assert (a[0] != b[0]).float().mean().item() < 1e-3
    if pool:
        assert (a[1] != b[1]).float().mean().item() < 1e-3
