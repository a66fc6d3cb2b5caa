"""The rounding-bound reference (tests/rounding_bound.py) on the CPU: its round-to-nearest-even against numpy's float16
and torch's bfloat16 conversions, and the interval's edges - ties to even, subnormals, overflow to inf, +-0 after ReLU,
padded channels."""
import numpy as np
import torch

import rounding_bound as rb

T = lambda a: torch.as_tensor(np.asarray(a, dtype=np.float64))


def _bf16_neighbours(y):
    """the bf16 values just below and just above the bf16 values y (float64)"""
    bits = torch.as_tensor(y, dtype=torch.float64).to(torch.float32).to(torch.bfloat16).view(torch.int16)
    step = torch.where(bits >= 0, 1, -1).to(torch.int16)
    up = (bits + step).view(torch.bfloat16).double()
    dn = (bits - step).view(torch.bfloat16).double()
    return torch.minimum(up, dn), torch.maximum(up, dn)


def _samples(rng, n, lo_exp, hi_exp):
    x = rng.standard_normal(n) * np.exp2(rng.integers(lo_exp, hi_exp, n))
    return np.concatenate([x, -x[:16], [0.0, -0.0]])


def test_rn_fp16_matches_numpy_everywhere():
    rng = np.random.default_rng(0)
    x = _samples(rng, 200000, -30, 17)                                   # subnormals ... overflow
    # exact midpoints between neighbouring fp16 values: ties to even, in the normal and the subnormal range
    h = np.unique(rng.integers(0, 0x7bff, 20000).astype(np.uint16)).view(np.float16).astype(np.float64)
    hn = np.nextafter(h.astype(np.float16), np.float16(np.inf)).astype(np.float64)
    mids = (h + hn) / 2
    x = np.concatenate([x, mids, -mids, [65504.0, 65519.99, 65520.0, 70000.0, -65520.0, 2.0 ** -25, 3 * 2.0 ** -26, 2.0 ** -26]])
    got = rb.rn(T(x), 'fp16').numpy()
    with np.errstate(over='ignore'):
        want = x.astype(np.float16).astype(np.float64)
    assert np.array_equal(got, want)
    assert np.array_equal(np.signbit(got), np.signbit(want))
    assert rb.rn(T([65519.99]), 'fp16').item() == 65504.0 and rb.rn(T([65520.0]), 'fp16').item() == np.inf
    assert rb.rn(T([-65520.0]), 'fp16').item() == -np.inf
    assert rb.rn(T([2.0 ** -25]), 'fp16').item() == 0.0                  # tie between 0 and the smallest subnormal: even
    assert rb.rn(T([3 * 2.0 ** -25]), 'fp16').item() == 2.0 ** -23       # tie between 1 and 2 subnormal steps: even


def test_rn_bf16_matches_torch_on_float32_inputs():
    rng = np.random.default_rng(1)
    x = _samples(rng, 200000, -140, 126).astype(np.float32)            # float32 subnormals included
    b = torch.as_tensor(rng.integers(1, 0x7f7f, 20000).astype(np.int16)).view(torch.bfloat16).double()
    _, bn = _bf16_neighbours(b)
    mids = ((b + bn) / 2).numpy().astype(np.float32)                     # bf16 midpoints are exact in float32
    x = np.concatenate([x, mids, -mids]).astype(np.float32)
    got = rb.rn(torch.as_tensor(x.astype(np.float64)), 'bf16')
    want = torch.as_tensor(x).to(torch.bfloat16).double()
    assert torch.equal(got, want)
    assert torch.equal(torch.signbit(got), torch.signbit(want))
    # float64 input one float32-ulp-below-half above a bf16 midpoint: a cast through float32 would round twice
    m = 1.0 + 2.0 ** -8 + 2.0 ** -40
    assert rb.rn(T([m]), 'bf16').item() == 1.0 + 2.0 ** -7


def test_interval_with_zero_delta_is_exactly_rn():
    rng = np.random.default_rng(2)
    for fmt in ('fp16', 'bf16'):
        v = T(rng.standard_normal(5000) * np.exp2(rng.integers(-20, 12, 5000)))
        lo, hi = rb.interval(v, torch.zeros_like(v), fmt, relu=True)
        r = rb.rn(torch.clamp(v, min=0), fmt)
        assert torch.equal(lo, r) and torch.equal(hi, r)
        pos = r > 0
        if fmt == 'fp16':
            rn16 = r.numpy().astype(np.float16)
            up = T(np.nextafter(rn16, np.float16(np.inf)))
            dn = T(np.nextafter(rn16, np.float16(-np.inf)))
        else:
            dn, up = _bf16_neighbours(r)
        for nb in (up, dn):
            ok = (nb >= lo) & (nb <= hi)
            assert not bool(ok[pos].any()), fmt


def test_check_edges_zero_padded_overflow_subnormal():
    z = T([0.0])
    one = T([1.0])
    # ReLU: a negative result admits +0 and -0 and nothing else
    for y in (0.0, -0.0):
        rep = rb.check(torch.tensor([y], dtype=torch.float16), T([-3.0]), T([4.0]), one, z)
        assert rep['bad'] == 0 and rep['sharp'] == 1.0
    rep = rb.check(torch.tensor([2.0 ** -24], dtype=torch.float16), T([-3.0]), T([4.0]), one, z)
    assert rep['bad'] == 1
    # padded channel: B = 0, scale = shift = 0 -> exactly 0
    rep = rb.check(torch.tensor([0.0, 2.0 ** -24], dtype=torch.float16), T([0.0, 0.0]), T([0.0, 0.0]), z, z)
    assert rep['bad'] == 1 and rep['first_bad']['index'] == 1
    # fp16 overflow: RN16 of a value >= 65520 is +inf; 65504 is wrong there, inf is wrong below 65504 + 16
    big = T([70000.0, 65519.0])
    rep = rb.check(torch.tensor([np.inf, 65504.0], dtype=torch.float16), big, T([1.0, 1.0]), one, z)
    assert rep['bad'] == 0
    rep = rb.check(torch.tensor([65504.0, np.inf], dtype=torch.float16), big, T([1.0, 1.0]), one, z)
    assert rep['bad'] == 2
    # NaN is never accepted
    assert rb.check(torch.tensor([np.nan], dtype=torch.float16), one, one, one, z)['bad'] == 1
    # fp16 subnormal result: exact subnormal accepted, its neighbour rejected when delta is tiny
    v = 5 * 2.0 ** -24
    rep = rb.check(torch.tensor([v], dtype=torch.float16), T([v]), T([v]), one, z, c_acc=0.0)
    assert rep['bad'] == 0 and rep['exact'] == 1.0
    rep = rb.check(torch.tensor([6 * 2.0 ** -24], dtype=torch.float16), T([v]), T([v]), one, z, c_acc=0.0)
    assert rep['bad'] == 1


def test_check_accepts_accumulation_error_within_c_acc_and_reports_ulps():
    rng = np.random.default_rng(3)
    n = 20000
    A = T(rng.standard_normal(n) * 4)
    B = A.abs() * 40                                                    # a typical ratio B / |A| for K ~ 5000
    scale, shift = T(rng.uniform(0.5, 1.5, n)), T(rng.standard_normal(n))
    for fmt, dt in (('fp16', torch.float16), ('bf16', torch.bfloat16)):
        # an accumulation error of c_acc * 2^-24 * B: still accepted
        Ae = A + 1.0 * rb.U24 * B * T(rng.choice([-1, 1], n))
        y = torch.clamp(scale * Ae + shift, min=0).float().to(dt)
        rep = rb.check(y, A, B, scale, shift, c_acc=1.0, fmt=fmt)
        assert rep['bad'] == 0 and rep['sharp'] >= 0.99, (fmt, rep)
        # one ulp off everywhere: rejected nearly everywhere it is not a clipped zero
        vr = torch.clamp(scale * A + shift, min=0)
        y1 = rb.rn(vr, fmt) + rb.quantum(rb.rn(vr, fmt), fmt)
        rep = rb.check(y1.to(dt), A, B, scale, shift, c_acc=1.0, fmt=fmt)
        assert rep['bad'] >= 0.98 * n and rep['max_ulp'] >= 1.0


def test_fp32_form_and_acc_ratio():
    A = T([1.0, -2.0, 0.0])
    B = T([3.0, 2.0, 0.0])
    y = (A + T([2.0 * rb.U24 * 3.0, -rb.U24, 0.0])).float()
    assert abs(rb.acc_ratio(y, A, B) - 2.0) < 1e-6
    assert rb.check(y, A, B, c_acc=2.0, relu=False)['bad'] == 0
    assert rb.check(y, A, B, c_acc=1.0, relu=False)['bad'] == 1
    assert rb.acc_ratio(torch.tensor([1e-30]), T([0.0]), T([0.0])) == np.inf


def test_exactness_catches_one_ulp_errors_a_loose_bound_admits():
    """with a c_acc large enough that one-ulp neighbours lie inside the interval, a kernel off by one ulp in a fifth of
    its outputs still fails through the exactly-rounded fraction; zeros do not count towards it"""
    import pytest
    rng = np.random.default_rng(4)
    n = 20000
    A = T(rng.standard_normal(n))
    B = A.abs() * 400
    one, z = T([1.0]), T([0.0])
    vr = torch.clamp(A, min=0)
    y = rb.rn(vr, 'fp16')
    rep = rb.check(y.to(torch.float16), A, B, one, z, c_acc=64.0)
    assert rep['bad'] == 0 and rep['exact_nz'] == 1.0 and rep['exact'] == 1.0
    rb.assert_ok(rep, 'exact')
    off = (torch.arange(n) % 5 == 0) & (y > 0)
    y1 = torch.where(off, y + rb.quantum(y, 'fp16'), y)
    rep = rb.check(y1.to(torch.float16), A, B, one, z, c_acc=64.0)
    assert rep['bad'] == 0 and 0.75 < rep['exact_nz'] < 0.85 and rep['exact'] > 0.85
    with pytest.raises(AssertionError):
        rb.assert_ok(rep, 'one ulp off in a fifth of the outputs')
