"""Thin torch-tensor wrappers over the dcb200 C ABI (include/dcb200.h).

torch is plumbing here: it owns device memory and the current stream; every
arithmetic op below is one call into libdcb200.so.  Nothing falls back to torch
or numpy arithmetic.
"""
import ctypes

import numpy as np
import torch

from .. import _native as nat
from .._native import c_int, c_ll, c_f, c_p, c_sz, ptr, stream_ptr, call

DT = {torch.float32: nat.DCB_F32, torch.bfloat16: nat.DCB_BF16, torch.float16: nat.DCB_F16}
c_ull = ctypes.c_ulonglong
c_uint = ctypes.c_uint


def _dt(t):
    return c_int(DT[t.dtype])


def _chk(t, dtype=None):
    assert t.is_cuda and t.is_contiguous(), 'dcb ops need contiguous CUDA tensors'
    if dtype is not None:
        assert t.dtype == dtype, (t.dtype, dtype)
    return t


# ---------------------------------------------------------------- projection (nf.py:115-130)
def proj_workspace_bytes(T, H, W):
    out = c_sz(0)
    call('dcb_proj_workspace_bytes', c_int(T), c_int(H), c_int(W), ctypes.byref(out))
    return out.value


def proj_mean_max(movie, mean, mx, workspace, floor_max_at_zero=False, variant=-1, t_splits=0):
    _chk(mean, torch.float32); _chk(mx, torch.float32)
    T, H, W = movie.shape
    if movie.dtype == torch.int16:        # the reference's raw TIFF frames: exact integer sums, half the bytes
        _chk(movie, torch.int16)
        call('dcb_proj_mean_max_i16', ptr(movie), c_int(T), c_int(H), c_int(W), ptr(mean), ptr(mx),
             c_int(int(floor_max_at_zero)), ptr(workspace),
             c_sz(workspace.numel() * workspace.element_size() if workspace is not None else 0), stream_ptr())
        return
    _chk(movie, torch.float32)
    call('dcb_proj_mean_max_f32_variant', ptr(movie), c_int(T), c_int(H), c_int(W), ptr(mean), ptr(mx),
         c_int(int(floor_max_at_zero)), ptr(workspace),
         c_sz(workspace.numel() * workspace.element_size() if workspace is not None else 0),
         c_int(variant), c_int(t_splits), stream_ptr())


def proj_accum_i16(chunk, sum_i64, max_i32):
    _chk(chunk, torch.int16); _chk(sum_i64, torch.int64); _chk(max_i32, torch.int32)
    Tc, H, W = chunk.shape
    call('dcb_proj_accum_i16', ptr(chunk), c_int(Tc), c_int(H), c_int(W), ptr(sum_i64), ptr(max_i32), stream_ptr())


def proj_accum_finalize(sum_i64, max_i32, T, mean, mx, floor_max_at_zero=False, bias=0):
    H, W = mean.shape
    call('dcb_proj_accum_finalize_biased', ptr(sum_i64), ptr(max_i32), c_int(T), c_int(H), c_int(W), c_int(int(bias)),
         ptr(mean), ptr(mx), c_int(int(floor_max_at_zero)), stream_ptr())


def standardize(x, out, stats=None):
    _chk(x, torch.float32); _chk(out, torch.float32)
    call('dcb_standardize_f32', ptr(x), c_ll(x.numel()), ptr(out), ptr(stats), stream_ptr())


# ---------------------------------------------------------------- contractions
def conv3x3_fwd(src0, src1, wgt, out, scale=None, shift=None, relu=False):
    N, H, W, C0 = src0.shape
    C1 = 0 if src1 is None else src1.shape[3]
    Cout = out.shape[3]
    call('dcb_conv3x3_fwd', _dt(src0), ptr(src0), c_int(C0), ptr(src1), c_int(C1), c_int(N), c_int(H), c_int(W),
         ptr(wgt), c_int(Cout), ptr(scale), ptr(shift), c_int(int(relu)), ptr(out), stream_ptr())


class ConvFusion(ctypes.Structure):
    _fields_ = [('head_kernel', c_p), ('head_bias', c_p), ('logit', c_p), ('prob', c_p), ('need_y', c_int),
                ('pool_out', c_p)]


def conv3x3_fwd_fused(src0, src1, wgt, out, scale=None, shift=None, relu=False, head_kernel=None, head_bias=None,
                      logit=None, prob=None, need_y=True, pool_out=None):
    """conv3x3 with the following max-pool and/or the softmax head folded into its epilogue."""
    N, H, W, C0 = src0.shape
    C1 = 0 if src1 is None else src1.shape[3]
    f = ConvFusion(ptr(head_kernel), ptr(head_bias), ptr(logit), ptr(prob), int(bool(need_y)), ptr(pool_out))
    call('dcb_conv3x3_fwd_fused', _dt(src0), ptr(src0), c_int(C0), ptr(src1), c_int(C1), c_int(N), c_int(H), c_int(W),
         ptr(wgt), c_int(out.shape[3]), ptr(scale), ptr(shift), c_int(int(relu)), ptr(out), ctypes.byref(f), stream_ptr())


def conv3x3_fwd_stats(src0, src1, wgt, out, sums_q, scale=None, shift=None, relu=False):
    """training forward: conv3x3 whose epilogue also accumulates the BatchNorm batch sums of the stored output into
    ``sums_q`` (int64 [2*Cout], 2^-20 fixed point, zeroed by the caller).  Returns True when the dispatched kernel did
    (else the caller runs its own statistics pass)."""
    N, H, W, C0 = src0.shape
    C1 = 0 if src1 is None else src1.shape[3]
    _chk(sums_q, torch.int64)
    done = c_int(0)
    call('dcb_conv3x3_fwd_stats', _dt(src0), ptr(src0), c_int(C0), ptr(src1), c_int(C1), c_int(N), c_int(H), c_int(W),
         ptr(wgt), c_int(out.shape[3]), ptr(scale), ptr(shift), c_int(int(relu)), ptr(out), ptr(sums_q), ctypes.byref(done),
         stream_ptr())
    return bool(done.value)


def convT2x2_fwd_stats(src, wgt, out, sums_q, scale=None, shift=None, relu=False):
    N, h, w, Cin = src.shape
    _chk(sums_q, torch.int64)
    done = c_int(0)
    call('dcb_convT2x2_fwd_stats', _dt(src), ptr(src), c_int(Cin), c_int(N), c_int(h), c_int(w), ptr(wgt), c_int(out.shape[3]),
         ptr(scale), ptr(shift), c_int(int(relu)), ptr(out), ptr(sums_q), ctypes.byref(done), stream_ptr())
    return bool(done.value)


def conv3x3_c1_fwd_stats(x, w, out, sums_q, scale=None, shift=None, relu=False):
    N, H, W = x.shape
    _chk(x, torch.float32); _chk(w, torch.float32); _chk(sums_q, torch.int64)
    done = c_int(0)
    call('dcb_conv3x3_c1_fwd_stats', _dt(out), ptr(x), c_int(N), c_int(H), c_int(W), ptr(w), c_int(out.shape[3]), ptr(scale),
         ptr(shift), c_int(int(relu)), ptr(out), ptr(sums_q), ctypes.byref(done), stream_ptr())
    return bool(done.value)


def conv3x3_dgrad(dy, wgt_dgrad, dx):
    """dy: [N,H,W,Cout] activation dtype (gradient w.r.t. the raw conv output); dx: fp32 [N,H,W,Cin]."""
    N, H, W, Cout = dy.shape
    _chk(dx, torch.float32)
    call('dcb_conv3x3_dgrad', _dt(dy), ptr(dy), c_int(Cout), c_int(N), c_int(H), c_int(W), ptr(wgt_dgrad),
         c_int(dx.shape[3]), ptr(dx), stream_ptr())


def convT2x2_fwd(src, wgt, out, scale=None, shift=None, relu=False):
    N, h, w, Cin = src.shape
    Cout = out.shape[3]
    call('dcb_convT2x2_fwd', _dt(src), ptr(src), c_int(Cin), c_int(N), c_int(h), c_int(w), ptr(wgt), c_int(Cout),
         ptr(scale), ptr(shift), c_int(int(relu)), ptr(out), stream_ptr())


def convT2x2_dgrad(dy, wgt, dx):
    _chk(dx, torch.float32)
    N, h, w, Cin = dx.shape
    Cout = dy.shape[3]
    call('dcb_convT2x2_dgrad', _dt(dy), ptr(dy), c_int(Cout), c_int(N), c_int(h), c_int(w), ptr(wgt), c_int(Cin),
         ptr(dx), stream_ptr())


def conv3x3_wgrad_workspace_bytes(dtype, N, H, W, Cin, Cout):
    out = c_sz(0)
    call('dcb_conv3x3_wgrad_workspace_bytes', c_int(DT[dtype]), c_int(N), c_int(H), c_int(W), c_int(Cin), c_int(Cout),
         ctypes.byref(out))
    return out.value


def conv3x3_wgrad(src0, src1, dy, dW, workspace):
    N, H, W, C0 = src0.shape
    C1 = 0 if src1 is None else src1.shape[3]
    Cout = dy.shape[3]
    _chk(dW, torch.float32)
    call('dcb_conv3x3_wgrad', _dt(src0), ptr(src0), c_int(C0), ptr(src1), c_int(C1), c_int(N), c_int(H), c_int(W),
         ptr(dy), c_int(Cout), ptr(dW), ptr(workspace), c_sz(workspace.numel() * workspace.element_size()), stream_ptr())


def convT2x2_wgrad_workspace_bytes(dtype, N, h, w, Cin, Cout):
    out = c_sz(0)
    call('dcb_convT2x2_wgrad_workspace_bytes', c_int(DT[dtype]), c_int(N), c_int(h), c_int(w), c_int(Cin), c_int(Cout),
         ctypes.byref(out))
    return out.value


def convT2x2_wgrad(x, dy, dW, workspace):
    N, h, w, Cin = x.shape
    Cout = dy.shape[3]
    call('dcb_convT2x2_wgrad', _dt(x), ptr(x), c_int(Cin), c_int(N), c_int(h), c_int(w), ptr(dy), c_int(Cout), ptr(dW),
         ptr(workspace), c_sz(workspace.numel() * workspace.element_size()), stream_ptr())


def conv3x3_c1_fwd(x, w, out, scale=None, shift=None, relu=False):
    """x: fp32 [N,H,W]; w: fp32 [3,3,1,Cout]; out: [N,H,W,Cout] in the activation dtype."""
    _chk(x, torch.float32); _chk(w, torch.float32)
    N, H, W = x.shape
    call('dcb_conv3x3_c1_fwd', _dt(out), ptr(x), c_int(N), c_int(H), c_int(W), ptr(w), c_int(out.shape[3]),
         ptr(scale), ptr(shift), c_int(int(relu)), ptr(out), stream_ptr())


def conv3x3_c1_wgrad_workspace_bytes(Cout):
    out = c_sz(0)
    call('dcb_conv3x3_c1_wgrad_workspace_bytes', c_int(Cout), ctypes.byref(out))
    return out.value


def conv3x3_c1_wgrad(x, dy, dW, workspace):
    N, H, W = x.shape
    call('dcb_conv3x3_c1_wgrad', _dt(dy), ptr(x), ptr(dy), c_int(N), c_int(H), c_int(W), c_int(dy.shape[3]), ptr(dW),
         ptr(workspace), c_sz(workspace.numel() * workspace.element_size()), stream_ptr())


def prep_conv3x3_weights(w, w_fwd, w_dgrad, dtype):
    _chk(w, torch.float32)
    Cin, Cout = w.shape[2], w.shape[3]
    call('dcb_prep_conv3x3_weights', c_int(DT[dtype]), ptr(w), c_int(Cin), c_int(Cout), ptr(w_fwd), ptr(w_dgrad),
         stream_ptr())


def prep_convT2x2_weights(w, w_fwd, w_dgrad, dtype):
    _chk(w, torch.float32)
    Cout, Cin = w.shape[2], w.shape[3]
    call('dcb_prep_convT2x2_weights', c_int(DT[dtype]), ptr(w), c_int(Cin), c_int(Cout), ptr(w_fwd), ptr(w_dgrad),
         stream_ptr())


# ---------------------------------------------------------------- BatchNorm
def prep_weights_batch(desc_dev, count, dtype):
    """desc_dev: int64 CUDA tensor [count, 5] (see dcb_prep_weights_batch)."""
    _chk(desc_dev, torch.int64)
    call('dcb_prep_weights_batch', c_int(DT[dtype]), ptr(desc_dev), c_int(count), stream_ptr())


def bn_fold(gamma, beta, mean, var, bias, scale, shift, eps=1e-3):
    call('dcb_bn_fold', ptr(gamma), ptr(beta), ptr(mean), ptr(var), ptr(bias), c_int(gamma.numel()), c_f(eps),
         ptr(scale), ptr(shift), stream_ptr())


def bn_stats(x, sums):
    C = x.shape[-1]
    call('dcb_bn_stats', _dt(x), ptr(x), c_ll(x.numel() // C), c_int(C), ptr(sums), stream_ptr())


def bn_finalize(sums, M, gamma, beta, momentum, moving_mean, moving_var, scale, shift, mean, rstd, eps=1e-3):
    call('dcb_bn_finalize', ptr(sums), c_ll(M), c_int(gamma.numel()), ptr(gamma), ptr(beta), c_f(eps), c_f(momentum),
         ptr(moving_mean), ptr(moving_var), ptr(scale), ptr(shift), ptr(mean), ptr(rstd), stream_ptr())


def bn_apply(x, scale, shift, y, relu=True, p_drop=0., seed=0, seed_dev=None, layer=0):
    C = x.shape[-1]
    call('dcb_bn_apply', _dt(x), ptr(x), c_ll(x.numel() // C), c_int(C), ptr(scale), ptr(shift), c_int(int(relu)),
         c_f(p_drop), c_ull(seed), ptr(seed_dev), c_uint(layer), ptr(y), stream_ptr())


def bn_finalize_apply(x, sums, M_total, gamma, beta, momentum, moving_mean, moving_var, scale, shift, mean, rstd, y,
                      relu=True, p_drop=0., seed=0, seed_dev=None, layer=0, eps=1e-3):
    C = x.shape[-1]
    call('dcb_bn_finalize_apply', _dt(x), ptr(x), c_ll(x.numel() // C), c_int(C), ptr(sums), c_ll(M_total), ptr(gamma),
         ptr(beta), c_f(eps), c_f(momentum), ptr(moving_mean), ptr(moving_var), ptr(scale), ptr(shift), ptr(mean), ptr(rstd),
         c_int(int(relu)), c_f(p_drop), c_ull(seed), ptr(seed_dev), c_uint(layer), ptr(y), stream_ptr())


def bn_bwd_reduce(dy, ldy, offy, x, scale, shift, mean, rstd, sums, p_drop=0., seed=0, seed_dev=None, layer=0):
    C = x.shape[-1]
    call('dcb_bn_bwd_reduce', _dt(x), ptr(dy), c_int(ldy), c_int(offy), ptr(x), c_ll(x.numel() // C), c_int(C),
         ptr(scale), ptr(shift), ptr(mean), ptr(rstd), c_f(p_drop), c_ull(seed), ptr(seed_dev), c_uint(layer),
         ptr(sums), stream_ptr())


def bn_bwd_apply(dy, ldy, offy, x, scale, shift, mean, rstd, sums, draw, dgamma, dbeta, p_drop=0., seed=0,
                 seed_dev=None, layer=0, M_total=0, dgb_scale=1.0):
    C = x.shape[-1]
    call('dcb_bn_bwd_apply', _dt(x), ptr(dy), c_int(ldy), c_int(offy), ptr(x), c_ll(x.numel() // C), c_int(C),
         ptr(scale), ptr(shift), ptr(mean), ptr(rstd), c_f(p_drop), c_ull(seed), ptr(seed_dev), c_uint(layer),
         ptr(sums), c_ll(M_total), c_f(dgb_scale), ptr(draw), ptr(dgamma), ptr(dbeta), stream_ptr())


class PeerExchange(ctypes.Structure):
    """dcb_peer_exchange_t"""
    _fields_ = [('world', c_int), ('rank', c_int), ('xchg', c_p * 8), ('flags', c_p * 8), ('slot_doubles', c_ll),
                ('slot', c_int), ('epoch_dev', c_p)]


def _peers_arg(peers, slot):
    if peers is None:
        return None
    px = PeerExchange()
    px.world, px.rank = peers['world'], peers['rank']
    for i in range(peers['world']):
        px.xchg[i] = peers['xchg'][i]
        px.flags[i] = peers['flags'][i]
    px.slot_doubles = peers['slot_doubles']
    px.slot = slot
    px.epoch_dev = peers['epoch_dev']
    return ctypes.byref(px)


def bn_train_workspace_bytes(C):
    out = c_sz(0)
    call('dcb_bn_train_workspace_bytes', c_int(C), ctypes.byref(out))
    return out.value


def bn_train_fwd(x, gamma, beta, momentum, moving_mean, moving_var, scale, shift, mean, rstd, y, workspace, sync,
                 relu=True, p_drop=0., seed=0, seed_dev=None, layer=0, pool_out=None, M_total=0, eps=1e-3, peers=None, slot=0):
    """single-launch training BatchNorm forward (+ReLU, dropout, optional 2x2 max-pool); sync: 4 zeroed int32 words"""
    C = x.shape[-1]
    N, H, W = (x.shape[0], x.shape[1], x.shape[2]) if x.dim() == 4 else (0, 0, 0)
    call('dcb_bn_train_fwd', _dt(x), ptr(x), c_ll(x.numel() // C), c_int(C), c_ll(M_total), ptr(gamma), ptr(beta), c_f(eps),
         c_f(momentum), ptr(moving_mean), ptr(moving_var), ptr(scale), ptr(shift), ptr(mean), ptr(rstd), c_int(int(relu)),
         c_f(p_drop), c_ull(seed), ptr(seed_dev), c_uint(layer), ptr(y), ptr(pool_out), c_int(N), c_int(H), c_int(W),
         ptr(workspace), c_sz(workspace.numel() * workspace.element_size()), ptr(sync), _peers_arg(peers, slot), stream_ptr())


def bn_train_fwd_sums(x, sums_q, gamma, beta, momentum, moving_mean, moving_var, scale, shift, mean, rstd, y, relu=True,
                      p_drop=0., seed=0, seed_dev=None, layer=0, pool_out=None, M_total=0, eps=1e-3, peers=None, slot=0):
    """training BatchNorm forward from known batch sums (int64, 2^-20 units: conv*_fwd_stats): one pass, no grid barrier"""
    C = x.shape[-1]
    N, H, W = (x.shape[0], x.shape[1], x.shape[2]) if x.dim() == 4 else (0, 0, 0)
    _chk(sums_q, torch.int64)
    call('dcb_bn_train_fwd_sums', _dt(x), ptr(x), c_ll(x.numel() // C), c_int(C), c_ll(M_total), ptr(sums_q), ptr(gamma),
         ptr(beta), c_f(eps), c_f(momentum), ptr(moving_mean), ptr(moving_var), ptr(scale), ptr(shift), ptr(mean), ptr(rstd),
         c_int(int(relu)), c_f(p_drop), c_ull(seed), ptr(seed_dev), c_uint(layer), ptr(y), ptr(pool_out), c_int(N), c_int(H),
         c_int(W), _peers_arg(peers, slot), stream_ptr())


def bn_train_bwd(dy, ldy, offy, x, scale, shift, mean, rstd, draw, dgamma, dbeta, workspace, sync, p_drop=0., seed=0,
                 seed_dev=None, layer=0, M_total=0, dgb_scale=1.0, peers=None, slot=0):
    C = x.shape[-1]
    call('dcb_bn_train_bwd', _dt(x), ptr(dy), c_int(ldy), c_int(offy), ptr(x), c_ll(x.numel() // C), c_int(C), c_ll(M_total),
         ptr(scale), ptr(shift), ptr(mean), ptr(rstd), c_f(p_drop), c_ull(seed), ptr(seed_dev), c_uint(layer), c_f(dgb_scale),
         ptr(draw), ptr(dgamma), ptr(dbeta), ptr(workspace), c_sz(workspace.numel() * workspace.element_size()), ptr(sync),
         _peers_arg(peers, slot), stream_ptr())


def bn_train_bwd_rank1(gpix, wd, x, scale, shift, mean, rstd, draw, dgamma, dbeta, workspace, sync, p_drop=0., seed=0,
                       seed_dev=None, layer=0, M_total=0, dgb_scale=1.0, peers=None, slot=0):
    """bn_train_bwd whose upstream gradient is the rank-1 product gpix[r] * wd[c] (head_loss_bwd_rank1)"""
    C = x.shape[-1]
    call('dcb_bn_train_bwd_rank1', _dt(x), ptr(gpix), ptr(wd), ptr(x), c_ll(x.numel() // C), c_int(C), c_ll(M_total),
         ptr(scale), ptr(shift), ptr(mean), ptr(rstd), c_f(p_drop), c_ull(seed), ptr(seed_dev), c_uint(layer), c_f(dgb_scale),
         ptr(draw), ptr(dgamma), ptr(dbeta), ptr(workspace), c_sz(workspace.numel() * workspace.element_size()), ptr(sync),
         _peers_arg(peers, slot), stream_ptr())


# ---------------------------------------------------------------- peer-mapped memory (csrc/peer.cu)
def peer_alloc(nbytes):
    """-> (device pointer, 64-byte IPC handle)"""
    p = c_p(0)
    h = (ctypes.c_ubyte * 64)()
    call('dcb_peer_alloc', c_sz(nbytes), ctypes.byref(p), h)
    return p.value, bytes(h)


def peer_open(handle):
    p = c_p(0)
    h = (ctypes.c_ubyte * 64).from_buffer_copy(handle)
    call('dcb_peer_open', h, ctypes.byref(p))
    return p.value


def peer_close(ptr_value):
    call('dcb_peer_close', c_p(ptr_value))


def peer_free(ptr_value):
    call('dcb_peer_free', c_p(ptr_value))


def counter_advance(counter):
    _chk(counter, torch.int64)
    call('dcb_counter_advance', ptr(counter), stream_ptr())


def flag_signal(flag_addrs, epoch, offset=0):
    """flag_addrs: list of raw device addresses (possibly peer-mapped); epoch: int64 CUDA tensor [1]"""
    arr = (c_p * len(flag_addrs))(*flag_addrs)
    call('dcb_flag_signal', arr, c_int(len(flag_addrs)), ptr(epoch), c_ll(offset), stream_ptr())


def flag_wait(flags_addr, n, epoch, offset=0, at_least=False):
    call('dcb_flag_wait', c_p(flags_addr), c_int(n), ptr(epoch), c_ll(offset), c_int(int(at_least)), stream_ptr())


def peer_allreduce_f64(vals, peers, slot):
    _chk(vals, torch.float64)
    call('dcb_peer_allreduce_f64', ptr(vals), c_int(vals.numel()), _peers_arg(peers, slot), stream_ptr())


# ---------------------------------------------------------------- pooling
def crop_batch(img_ptrs, mask_ptrs, widths, desc, window, x_out, y_out):
    """tables: int64 [D], int64 [D], int32 [D]; desc int32 [B, 12]; x_out fp32 [B, n, n]; y_out uint8 [B, n, n]"""
    call('dcb_crop_batch', ptr(img_ptrs), ptr(mask_ptrs), ptr(widths), ptr(desc), c_int(desc.shape[0]), c_int(window),
         ptr(x_out), ptr(y_out), stream_ptr())


def upsample2x(x, y, p_drop=0., seed=0, seed_dev=None, layer=0):
    N, h, w, C = x.shape
    call('dcb_upsample2x', _dt(x), ptr(x), c_int(N), c_int(h), c_int(w), c_int(C), c_f(p_drop), c_ull(seed), ptr(seed_dev),
         c_uint(layer), ptr(y), stream_ptr())


def upsample2x_bwd(dy, ldy, offy, dx, p_drop=0., seed=0, seed_dev=None, layer=0):
    N, h, w, C = dx.shape
    call('dcb_upsample2x_bwd', ptr(dy), c_int(ldy), c_int(offy), c_int(N), c_int(h), c_int(w), c_int(C), c_f(p_drop),
         c_ull(seed), ptr(seed_dev), c_uint(layer), ptr(dx), stream_ptr())


def maxpool2x2(x, y):
    N, H, W, C = x.shape
    call('dcb_maxpool2x2', _dt(x), ptr(x), c_int(N), c_int(H), c_int(W), c_int(C), ptr(y), stream_ptr())


def pool_bwd_add(skipgrad, lds, offs, y, pooled, dpool, out):
    N, H, W, C = y.shape
    call('dcb_pool_bwd_add', _dt(y), ptr(skipgrad), c_int(lds), c_int(offs), ptr(y), ptr(pooled), ptr(dpool),
         c_int(N), c_int(H), c_int(W), c_int(C), ptr(out), stream_ptr())


# ---------------------------------------------------------------- head / loss
def head_fwd(x, w, b, logit, prob):
    C = x.shape[-1]
    call('dcb_head_fwd', _dt(x), ptr(x), c_ll(x.numel() // C), c_int(C), ptr(w), ptr(b), ptr(logit), ptr(prob),
         stream_ptr())


def head_loss_fwd(x, w, b, yt, prob, sums):
    C = x.shape[-1]
    _chk(yt, torch.uint8)
    call('dcb_head_loss_fwd', _dt(x), ptr(x), c_ll(x.numel() // C), c_int(C), ptr(w), ptr(b), ptr(yt), ptr(prob),
         ptr(sums), stream_ptr())


def head_loss_bwd(x, w, yt, prob, sums, loss_id, dx, dwb_accum, dw_out, metrics_out, M_total=0):
    C = x.shape[-1]
    call('dcb_head_loss_bwd', _dt(x), ptr(x), c_ll(x.numel() // C), c_int(C), ptr(w), ptr(yt), ptr(prob), ptr(sums),
         c_int(loss_id), c_ll(M_total), ptr(dx), ptr(dwb_accum), ptr(dw_out), ptr(metrics_out), stream_ptr())


def head_loss_bwd_rank1(x, w, yt, prob, sums, loss_id, gpix, wd_out, dwb_accum, dw_out, metrics_out, M_total=0):
    """head_loss_bwd that writes the two factors of the rank-1 gradient dL/dx[m][c] = gpix[m] * wd[c] instead of dL/dx
    (32 input channels)"""
    C = x.shape[-1]
    _chk(gpix, torch.float32); _chk(wd_out, torch.float32)
    call('dcb_head_loss_bwd_rank1', _dt(x), ptr(x), c_ll(x.numel() // C), c_int(C), ptr(w), ptr(yt), ptr(prob), ptr(sums),
         c_int(loss_id), c_ll(M_total), ptr(gpix), ptr(wd_out), ptr(dwb_accum), ptr(dw_out), ptr(metrics_out), stream_ptr())


# ---------------------------------------------------------------- TTA
def tta_make_batch(s, S, first, count, out):
    _chk(s, torch.float32)
    hs, ws = s.shape
    call('dcb_tta_make_batch', _dt(out), ptr(s), c_int(hs), c_int(ws), c_int(S), c_int(first), c_int(count), ptr(out),
         stream_ptr())


def tta_combine(probs, S, hs, ws, threshold, n_aug, act, mask):
    _chk(probs, torch.float32); _chk(mask, torch.uint8)
    call('dcb_tta_combine', ptr(probs), c_int(S), c_int(hs), c_int(ws), c_f(threshold), c_int(n_aug), ptr(act),
         ptr(mask), stream_ptr())


def tile_make_batch(s, T, origins_y, origins_x, tile_first, n_tiles, first, count, out):
    """the tiles tile_first.. of a plan (device int32 origins per dimension) under transforms first..first+count-1 ->
    out [n_tiles * count, T, T]"""
    _chk(s, torch.float32); _chk(origins_y, torch.int32); _chk(origins_x, torch.int32)
    hs, ws = s.shape
    call('dcb_tile_make_batch', _dt(out), ptr(s), c_int(hs), c_int(ws), c_int(T), ptr(origins_y), ptr(origins_x),
         c_int(origins_y.numel()), c_int(origins_x.numel()), c_int(tile_first), c_int(n_tiles), c_int(first), c_int(count),
         ptr(out), stream_ptr())


def tile_combine(probs, T, origins_y, origins_x, cuts_y, cuts_x, tile_first, n_tiles, threshold, n_aug, act, mask):
    """act / mask [hs, ws] at the pixels owned by the tiles tile_first..tile_first+n_tiles-1 of the plan"""
    _chk(probs, torch.float32); _chk(mask, torch.uint8)
    for t in (origins_y, origins_x, cuts_y, cuts_x):
        _chk(t, torch.int32)
    hs, ws = mask.shape
    call('dcb_tile_combine', ptr(probs), c_int(T), c_int(hs), c_int(ws), ptr(origins_y), ptr(origins_x),
         ptr(cuts_y if cuts_y.numel() else None), ptr(cuts_x if cuts_x.numel() else None), c_int(origins_y.numel()),
         c_int(origins_x.numel()), c_int(tile_first), c_int(n_tiles), c_f(threshold), c_int(n_aug), ptr(act), ptr(mask),
         stream_ptr())


# ---------------------------------------------------------------- region scoring (csrc/regions.cu)
# An image table is an int64 numpy array [n, 8] of {data pointer, H, W, row stride, column stride, kind, 0, 0} (strides in
# elements; kind 0 uint8 nonzero, 1 fp32 / 2 fp64 round(p) != 0); the calls take it on the host and on the device.
def _h_desc(h_desc):
    assert h_desc.dtype == np.int64 and h_desc.ndim == 2 and h_desc.shape[1] == 8 and h_desc.flags.c_contiguous
    return h_desc.ctypes.data_as(c_p)


def nf_score_workspace_bytes(h_desc):
    """-> (workspace bytes of label_regions / nf_score for this table, capacity of region_info in rows)"""
    nbytes, cap = c_sz(0), c_ll(0)
    call('dcb_nf_score_workspace_bytes', _h_desc(h_desc), c_int(h_desc.shape[0]), ctypes.byref(nbytes), ctypes.byref(cap))
    return nbytes.value, cap.value


def label_regions(desc, h_desc, labels, region_base, workspace):
    """labels int32 [sum H*W] (scipy.ndimage.label numbering, 8-connected), region_base int32 [n + 1]"""
    _chk(desc, torch.int64); _chk(labels, torch.int32); _chk(region_base, torch.int32); _chk(workspace, torch.uint8)
    call('dcb_label_regions', ptr(desc), _h_desc(h_desc), c_int(h_desc.shape[0]), ptr(labels), ptr(region_base),
         ptr(workspace), c_sz(workspace.numel()), stream_ptr())


def nf_score(desc, h_desc, region_base, region_info, workspace):
    """(truth, prediction) pairs as rows 2p, 2p+1 of the table -> region_base int32 [n + 1], region_info int32 [cap, 3]
    = {pixel count, matched prediction region of the pair or -1, overlap pixels}"""
    _chk(desc, torch.int64); _chk(region_base, torch.int32); _chk(region_info, torch.int32); _chk(workspace, torch.uint8)
    call('dcb_nf_score', ptr(desc), _h_desc(h_desc), c_int(h_desc.shape[0] // 2), ptr(region_base), ptr(region_info),
         ptr(workspace), c_sz(workspace.numel()), stream_ptr())


def mask_summary_workspace_bytes(n, H, W):
    out = c_sz(0)
    call('dcb_mask_summary_workspace_bytes', c_int(n), c_int(H), c_int(W), ctypes.byref(out))
    return out.value


def mask_summary(masks, out, workspace):
    """masks [n, H, W] (int8, uint8 or bool) -> out uint8 [H, W]: the reference's _summarize_mask"""
    _chk(masks); _chk(out, torch.uint8)
    assert masks.element_size() == 1, masks.dtype
    n, H, W = masks.shape
    call('dcb_mask_summary', ptr(masks), c_int(n), c_int(H), c_int(W), ptr(out), ptr(workspace),
         c_sz(workspace.numel() if workspace is not None else 0), stream_ptr())


def orient_pad(s, k, out):
    """out [H, W] = np.pad(f_k(s), ((0, H - hf), (0, W - wf)), 'reflect'), f_k = (identity, fliplr, flipud, rot90 1/2/3)[k]"""
    _chk(s, torch.float32); _chk(out, torch.float32)
    call('dcb_orient_pad_f32', ptr(s), c_int(s.shape[0]), c_int(s.shape[1]), c_int(k), c_int(out.shape[0]),
         c_int(out.shape[1]), ptr(out), stream_ptr())


# ---------------------------------------------------------------- optimiser
def adam_step(p, g, m, v, lr_t=0., lr_t_dev=None, beta1=0.9, beta2=0.999, eps=1e-8):
    call('dcb_adam_step', ptr(p), ptr(g), ptr(m), ptr(v), c_ll(p.numel()), c_f(lr_t), ptr(lr_t_dev), c_f(beta1),
         c_f(beta2), c_f(eps), stream_ptr())


def step_advance(state, lr, beta1, beta2, lr_t_out):
    call('dcb_step_advance', ptr(state), c_f(lr), c_f(beta1), c_f(beta2), ptr(lr_t_out), stream_ptr())


def cast_from_f32(x, out):
    call('dcb_cast_from_f32', _dt(out), ptr(x), c_ll(x.numel()), ptr(out), stream_ptr())


def cast_to_f32(x, out):
    call('dcb_cast_to_f32', _dt(x), ptr(x), c_ll(x.numel()), ptr(out), stream_ptr())
