"""ctypes binding of libdcb200.so (the C ABI declared in include/dcb200.h).

There is no CPU fallback: if the library is missing or a call fails, this module
raises.  ``lib()`` loads lazily so that importing ``deepcalcium`` works on a box
without a GPU (the host logic and the symbol-export tests run there).
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, '_lib', 'libdcb200.so')

_lib = None

c_int = ctypes.c_int
c_ll = ctypes.c_longlong
c_f = ctypes.c_float
c_d = ctypes.c_double
c_p = ctypes.c_void_p
c_sz = ctypes.c_size_t

DCB_F32, DCB_BF16, DCB_F16 = 0, 1, 2
# dcb_policy_key (include/dcb200.h)
POLICY_KEYS = {'flat': 0, 'strip': 1, 'fold': 2, 'nsplit': 3, 'swap_min_cout': 4, 'wgrad_strip': 5, 'bn_ctas_per_sm': 6,
               'proj_i16_splits': 7, 'splitk': 8, 'fused_bn': 9, 'tma_store': 10, 'bn_slab': 11, 'pdl': 12, 'pair': 13}
LOSS_IDS = {'binary_crossentropy': 0, 'weighted_binary_crossentropy': 1, 'dice_loss': 2, 'dicesq_loss': 3}


class DcbError(RuntimeError):
    pass


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise DcbError('libdcb200.so not built (%s); run `python deep-calcium_b200/build.py` or '
                           '__graft_entry__.build() - there is no CPU fallback' % LIB_PATH)
        _lib = ctypes.CDLL(LIB_PATH)
        _lib.dcb_last_error.restype = ctypes.c_char_p
        _lib.dcb_launch_count.restype = ctypes.c_ulonglong
        _lib.dcb_last_kernel.restype = ctypes.c_char_p
    return _lib


def check(status, what=''):
    if status != 0:
        msg = lib().dcb_last_error()
        raise DcbError('%s failed with status %d: %s' % (what or 'dcb call', status,
                                                        msg.decode() if msg else '?'))


def ptr(t):
    """Device pointer of a torch tensor (or None)."""
    if t is None:
        return c_p(0)
    return c_p(t.data_ptr())


def stream_ptr(device=None):
    """cudaStream_t of torch's current stream on `device` (default: the current device)."""
    import torch
    return c_p(torch.cuda.current_stream(device).cuda_stream)


def call(name, *args):
    fn = getattr(lib(), name)
    check(fn(*args), name)


def launch_count():
    return int(lib().dcb_launch_count())


def set_policy(**kw):
    """dcb_set_policy for each keyword (names in POLICY_KEYS), e.g. set_policy(flat=2, strip=0)."""
    for k, v in kw.items():
        check(lib().dcb_set_policy(c_int(POLICY_KEYS[k]), c_int(int(v))), 'dcb_set_policy')


def get_policy(name):
    out = c_int(0)
    check(lib().dcb_get_policy(c_int(POLICY_KEYS[name]), ctypes.byref(out)), 'dcb_get_policy')
    return out.value


def reset_policy():
    check(lib().dcb_reset_policy(), 'dcb_reset_policy')


class policy(object):
    """Context manager: pin a dispatch policy for the enclosed calls, restore the previous values afterwards."""

    def __init__(self, **kw):
        self.kw = kw

    def __enter__(self):
        self.saved = {k: get_policy(k) for k in self.kw}
        set_policy(**self.kw)
        return self

    def __exit__(self, *exc):
        set_policy(**self.saved)
        return False


def last_kernel():
    """name of the kernel variant the last dcb_conv* / dcb_*wgrad / BatchNorm call of this thread dispatched to"""
    s = lib().dcb_last_kernel()
    return s.decode() if s else ''


def require_cuda():
    import torch
    if not torch.cuda.is_available():
        raise DcbError('deepcalcium (B200 build) needs a CUDA device; there is no CPU fallback')
    lib()
