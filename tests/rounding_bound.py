"""Rounding-bound reference for one layer of the 16-bit (and fp32) inference kernels.

A layer computes y = [relu](scale * A + shift), A = sum(x * w), from stored 16-bit operands x, w and fp32 scale / shift.
Products of 16-bit values are exact in float64, so float64 gives A (and B = sum(|x| * |w|)) to 2^-53 relative.  A
correct kernel accumulates A in fp32 to within c_acc * 2^-24 * B, applies the epilogue FMA with one more fp32 rounding
and rounds the result to nearest-even into the output format.  Rounding is monotone, so the stored y must satisfy

    RN16(relu(v - d)) <= y <= RN16(relu(v + d)),   v = scale * A + shift,
    d = |scale| * c_acc * 2^-24 * B + 2^-24 * (|scale * A| + |shift|).

fp32 outputs (dgrad, wgrad, the fp32 check mode) drop the RN16 step.  Everything here works on float64 torch tensors on
any device (the layer walk keeps 8 x 512^2 x 64-channel tensors on the GPU).
"""
import torch

U24 = 2.0 ** -24

# c_acc: the largest |y - A| / (2^-24 * B) measured through the paths that expose the fp32 accumulator, over the
# conv cases of tests/test_gpu_ops.py and the padded / tiled layer shapes, on an NVIDIA B200 (1000 W power limit),
# with ~1.5x headroom.
# tcgen05.mma with bf16 / fp16 operands, measured through dcb_conv3x3_dgrad (the forward kernels with fp32 output), every
# dispatch variant, contraction length K = 9 * channels up to 4608: generic 10.5 (bf16) / 11.9 (fp16), generic_swap
# 6.1 / 6.9, flat 5.6 / 8.3, strip 5.1 / 6.3, strip_swap 5.1 / 6.1, strip_fold and strip_pair 4.8 / 6.2.  It grows with
# K: at K = 13824 (1536 channels) flat 21.1 / 23.3, generic 20.2 / 21.3, i.e. about 0.2 sqrt(K).  c_acc_tc(K) is
# 1.5x that, and at least 18.
C_ACC_TC = 18.0


def c_acc_tc(K):
    return max(C_ACC_TC, 0.3 * K ** 0.5)


# tcgen05.mma weight-gradient kernels (bf16 only): wgrad 2.6, wgrad_strip 2.3 on the unit cases, wgrad 5.4 over
# 32768 pixels.
C_ACC_WGRAD = 8.0
# CUDA-core fp32 check-mode kernels (tapgemm_f32.cu): forward 1.15, dgrad 1.25 on the unit cases; the layer walk's
# enc0b, up1 and up0 at 512^2 need up to ~4.1.
C_ACC_F32 = 6.0
# first-layer kernel (conv3x3_c1: fp32 input and weights, K = 9): the textbook bound K, far below a 16-bit ulp
C_ACC_C1 = 9.0
# (explicit mantissa bits, minimum normal exponent, maximum exponent)
FORMATS = {'fp16': (10, -14, 15), 'bf16': (7, -126, 127), 'fp32': (23, -126, 127)}
TORCH_FORMAT = {torch.float16: 'fp16', torch.bfloat16: 'bf16', torch.float32: 'fp32'}


def quantum(x, fmt):
    """spacing of format ``fmt`` at |x| (the ulp of the binade of x; the subnormal spacing below the normal range)"""
    mant, emin, _ = FORMATS[fmt]
    _, e = torch.frexp(x.abs())                 # |x| = m * 2^e, 0.5 <= m < 1  ->  binade exponent e - 1
    e = torch.clamp(e - 1, min=emin)
    return torch.ldexp(torch.ones_like(x), e - mant)


def rn(x, fmt):
    """round-to-nearest-even of float64 ``x`` into ``fmt`` (values as float64; +-inf past the largest finite value).
    Direct from float64: torch's float64 -> bfloat16 cast goes through float32 and can round twice."""
    x = x.to(torch.float64)
    mant, _, emax = FORMATS[fmt]
    q = quantum(x, fmt)
    y = torch.round(x / q) * q                  # x / q is exact (power-of-two scaling); torch.round is half-to-even
    big = (2.0 - 2.0 ** -mant) * 2.0 ** emax
    y = torch.where(y.abs() > big, torch.copysign(torch.full_like(y, float('inf')), y), y)
    return torch.where(torch.isfinite(x), y, x)


def _relu(t, relu):
    return torch.clamp(t, min=0.0) if relu else t


def interval(v, delta, fmt, relu=True):
    """[lo, hi]: every value a correct kernel may store for exact result v with accumulation error at most delta"""
    lo, hi = _relu(v - delta, relu), _relu(v + delta, relu)
    if fmt != 'fp32':
        lo, hi = rn(lo, fmt), rn(hi, fmt)
    return lo, hi


def delta(A, B, scale, shift, c_acc):
    return scale.abs() * (c_acc * U24) * B + U24 * ((scale * A).abs() + shift.abs())


def check(y, A, B, scale=None, shift=None, c_acc=C_ACC_TC, relu=True, fmt=None):
    """y: the stored output (any float dtype); A, B: float64 of y's shape; scale / shift: float64 broadcastable to it
    (None = 1 / 0).  Returns a report dict: n, bad (elements outside the interval), exact (fraction equal to
    RN16(v)), exact_nz (the same over the outputs whose RN16(v) is not zero), max_ulp (largest |y - v| in ulps of the
    output format), median_delta_ulp, sharp (fraction of elements whose interval is a single value or whose d is below
    1/4 ulp)."""
    fmt = fmt or TORCH_FORMAT[y.dtype]
    if scale is None:
        scale = torch.ones((), dtype=torch.float64, device=A.device)
    if shift is None:
        shift = torch.zeros((), dtype=torch.float64, device=A.device)
    y = y.to(torch.float64)
    v = scale * A + shift
    d = delta(A, B, scale, shift, c_acc)
    lo, hi = interval(v, d, fmt, relu)
    inside = (y >= lo) & (y <= hi)              # -0 == +0: both zeros pass where 0 is admitted; NaN never passes
    vr = _relu(v, relu)
    q = quantum(vr, fmt)
    d_ulp = d / q
    err_ulp = (y - vr).abs() / q
    want = vr if fmt == 'fp32' else rn(vr, fmt)
    hit, nz = y == want, want != 0
    n_nz = int(nz.sum())
    return dict(n=y.numel(), bad=int((~inside).sum()), exact=float(hit.double().mean()),
                exact_nz=float((hit & nz).sum()) / n_nz if n_nz else 1.0,
                max_ulp=float(err_ulp.max()) if y.numel() else 0.0, median_delta_ulp=float(d_ulp.median()) if y.numel() else 0.0,
                sharp=float(((lo == hi) | (d_ulp < 0.25)).double().mean()), first_bad=_first_bad(inside, y, lo, hi))


def _first_bad(inside, y, lo, hi):
    if bool(inside.all()):
        return None
    i = int((~inside).reshape(-1).nonzero()[0])
    return dict(index=i, y=float(y.reshape(-1)[i]), lo=float(lo.reshape(-1)[i]), hi=float(hi.reshape(-1)[i]))


def acc_ratio(y, A, B):
    """largest |y - A| / (2^-24 * B) of an fp32 output with no epilogue: the c_acc this tensor shows (0 where B = 0 and
    y == A; inf where B = 0 and y != A)"""
    err = (y.to(torch.float64) - A).abs()
    r = err / (U24 * B)
    r = torch.where(err == 0, torch.zeros_like(r), r)
    return float(r.max()) if r.numel() else 0.0


# Teeth.  The bound alone catches a one-ulp error only where d < 1/2 ulp.  With the measured c_acc, d < 1/4 ulp holds
# for 0.96 - 0.99 of the outputs of most fp16 layers, but only for 0.79 - 0.90 of them at K = 9216 - 13824 (the
# 1024-channel botb, the 1536-channel concats).  Few outputs carry that much accumulation error, though: the kernels
# store exactly RN16(v) in at least 0.948 of the non-zero outputs of every fp16 tensor checked, and 0.993 in bf16.  So
# every checked 16-bit tensor must also be exactly rounded in at least EXACT_MIN of its non-zero outputs: a kernel off
# by one ulp in more than a tenth of its outputs fails, whatever the contraction length.  'sharp' (the fraction with a
# single admissible value or d < 1/4 ulp) is reported next to it.
EXACT_MIN = 0.9


def assert_ok(rep, what, exact=True):
    assert rep['bad'] == 0, '%s: %d of %d outputs outside the rounding bound, first %s' % (what, rep['bad'], rep['n'], rep['first_bad'])
    if exact:
        assert rep['exact_nz'] >= EXACT_MIN, '%s: only %.4f of the non-zero outputs are exactly RN16(v) (sharp %.4f)' % (
            what, rep['exact_nz'], rep['sharp'])
