"""Tensor-level wrappers over the C-ABI (include/msg_b200.h).  PyTorch is used for device memory
and streams only; every computation below is a hand-written sm_100a kernel in csrc/.

Activations are NHWC tensors ``[N, H, W, C]`` (contiguous) of dtype float32 or bfloat16.
"""
import ctypes

import torch

from . import _lib
from ._lib import (ACT_LRELU, ACT_NONE, ACT_RELU, ACT_TANH, CONV_ACCUM, CONV_FORCE_GATHER, CONV_FORCE_SIMT, CONV_IN_NORM,
                   CONV_OUT_NCHW_F32, CONV_STATS, PACK_CONVT_PHASES, PACK_DGRAD_S1, PACK_FWD, ConvDesc)

_DT = {torch.float32: _lib.F32, torch.bfloat16: _lib.BF16}


def _dt(t):
    try:
        return _DT[t.dtype]
    except KeyError:
        raise _lib.MsgError(f"unsupported dtype {t.dtype}; the path computes in float32 or bfloat16")


def _p(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)
_raw_device = getattr(torch._C, "_cuda_getDevice", None)


def _stream():
    """Raw handle of torch's current stream on the current device.  torch.cuda.current_stream() builds a Python Stream
    object (~15 us, a quarter of the host time of a launch-bound train step); the raw accessor costs ~0.3 us.
    The C-ABI launches on the CURRENT device (it never calls cudaSetDevice): `_dev` below refuses tensors that live on
    another device, and the module-level entry points (EnhancedGenerator.forward, ...) run under
    ``torch.cuda.device(x.device)``."""
    if _raw_stream is not None and _raw_device is not None:
        return ctypes.c_void_p(_raw_stream(_raw_device()))
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _dev(t):
    if not t.is_cuda:
        raise _lib.MsgError("msg_b200 ops need CUDA tensors: there is no CPU fallback in this package")
    idx = t.device.index
    cur = _raw_device() if _raw_device is not None else torch.cuda.current_device()
    if idx != cur:
        # a launch on the current device with another device's pointers = illegal address at best, silent peer traffic at worst
        raise _lib.MsgError(f"msg_b200 op on a cuda:{idx} tensor while the current device is cuda:{cur}: the kernels launch "
                            f"on the current device -- wrap the call in `with torch.cuda.device({idx}):`")
    _lib.require_device(idx)


def _aff(affine):
    """(gamma, beta, img_stride) of an optional InstanceNorm affine -> C-ABI arguments (include/msg_b200.h); gamma / beta are
    fp32 device tensors whose first element is that of image 0, channel 0 of the site."""
    if affine is None:
        return None, None, 0
    g, b, stride = affine
    return _p(g), _p(b), int(stride)


def conv_raw(desc, x, w, bias, y, stats=None, in_stats=None, in_affine=None):
    if in_affine is None:
        _lib.call("msg_conv2d", ctypes.byref(desc), _p(x), _p(w), _p(bias), _p(y), _p(stats), _p(in_stats), _stream())
    else:
        _lib.call("msg_conv2d_affine", ctypes.byref(desc), _p(x), _p(w), _p(bias), _p(y), _p(stats), _p(in_stats), *_aff(in_affine),
                  _stream())


def make_desc(dt, N, Hi, Wi, Ci_total, ci_off, Cin, Ho, Wo, Co_total, co_off, Cout, Hg, Wg, KH, KW,
              in_stride, pad_h, pad_w, dil, out_stride=1, out_off_h=0, out_off_w=0, act=ACT_NONE,
              flags=0, in_act=ACT_NONE):
    return ConvDesc(dt, N, Hi, Wi, Ci_total, ci_off, Cin, Ho, Wo, Co_total, co_off, Cout, Hg, Wg, KH, KW,
                    in_stride, pad_h, pad_w, dil, out_stride, out_off_h, out_off_w, act, flags, in_act)


def pack_weight(w, mode, dtype, sigma=None):
    """fp32 master weight [d0, d1, KH, KW] -> packed operand (flat tensor of `dtype`)."""
    _dev(w)
    w = w.detach()
    assert w.dtype == torch.float32 and w.is_contiguous()
    d0, d1, KH, KW = w.shape
    out = torch.empty(w.numel(), device=w.device, dtype=dtype)
    _lib.call("msg_pack_conv_weight", _p(w), d0, d1, KH, KW, mode, _DT[dtype], _p(sigma), _p(out), _stream())
    return out


def unpack_wgrad(dw_packed, shape, mode, dw):
    d0, d1, KH, KW = shape
    _lib.call("msg_unpack_conv_wgrad", _p(dw_packed), d0, d1, KH, KW, mode, _p(dw), _stream())


class ConvGeom:
    """Geometry of one convolution of the path + the launches for forward / dgrad / wgrad.

    kind 'conv'  : nn.Conv2d(Cin, Cout, k, stride, pad, dilation) weight [Cout, Cin, k, k]
    kind 'convT' : nn.ConvTranspose2d(Cin, Cout, 4, 2, 1)          weight [Cin, Cout, 4, 4]
                   (four sub-pixel phases, each a 2x2 gather conv writing every other pixel)
    """

    def __init__(self, kind, Cin, Cout, k, stride=1, pad=0, dil=1):
        assert kind in ("conv", "convT")
        if kind == "convT":
            assert (k, stride, pad, dil) == (4, 2, 1, 1)
        else:
            assert stride == 1 or (k, stride, pad, dil) == (4, 2, 1, 1), "strided conv: only 4x4 s2 p1"
        self.kind, self.Cin, self.Cout, self.k, self.stride, self.pad, self.dil = kind, Cin, Cout, k, stride, pad, dil

    # ---- shapes
    def out_hw(self, Hi, Wi):
        if self.kind == "convT":
            return 2 * Hi, 2 * Wi
        e = self.dil * (self.k - 1)
        return (Hi + 2 * self.pad - e - 1) // self.stride + 1, (Wi + 2 * self.pad - e - 1) // self.stride + 1

    def weight_shape(self):
        if self.kind == "convT":
            return (self.Cin, self.Cout, 4, 4)
        return (self.Cout, self.Cin, self.k, self.k)

    # ---- packing
    def pack_fwd(self, w, dtype, sigma=None):
        return pack_weight(w, PACK_CONVT_PHASES if self.kind == "convT" else PACK_FWD, dtype, sigma)

    def pack_dgrad(self, w, dtype, sigma=None):
        if self.kind == "convT":
            return pack_weight(w, PACK_FWD, dtype, sigma)  # [Cin][Cout][4][4] read as OIHW with O=Cin
        if self.stride == 2:
            return pack_weight(w, PACK_CONVT_PHASES, dtype, sigma)  # conv weight read as convT weight
        return pack_weight(w, PACK_DGRAD_S1, dtype, sigma)

    def fused_in_norm_ok(self, x, wp):
        """True when msg_conv2d would run this conv WITH a fused input InstanceNorm on the TMA + tcgen05 kernel
        (1x1 stride-1 convs, bf16, Cin % 64 == 0, tiles inside one image); otherwise the caller keeps the separate
        IN-apply pass (the only other engine with a fused input norm is the SIMT parity engine)."""
        if self.kind != "conv" or self.k != 1 or self.stride != 1:
            return False
        N, Hi, Wi, Ci_total = x.shape
        key = (N, Hi, Wi, Ci_total, x.dtype)
        hit = self._fuse_cache.get(key) if hasattr(self, "_fuse_cache") else None
        if hit is None:
            if not hasattr(self, "_fuse_cache"):
                self._fuse_cache = {}
            d = make_desc(_dt(x), N, Hi, Wi, Ci_total, 0, self.Cin, Hi, Wi, self.Cout, 0, self.Cout, Hi, Wi, 1, 1, 1, 0, 0,
                          1, 1, 0, 0, ACT_NONE, CONV_IN_NORM, ACT_RELU)
            # pointers only matter for their alignment: fresh torch allocations are 256-byte aligned like x / wp
            hit = _lib.load().msg_conv2d_path(ctypes.byref(d), _p(x), _p(wp), _p(x)) == 2
            self._fuse_cache[key] = hit
        return hit

    # ---- launches
    def forward(self, x, wp, bias, out=None, co_off=0, stats=None, act=ACT_NONE, in_stats=None,
                in_act=ACT_NONE, ci_off=0, nchw_out=None, extra_flags=0, in_affine=None):
        """x: [N,Hi,Wi,Ci_total].  Writes channels [co_off, co_off+Cout) of `out` [N,Ho,Wo,Co_total]
        (allocated if None).  nchw_out: fp32 [N,Cout,Ho,Wo] tensor to write instead (final image).
        in_affine: (gamma, beta, img_stride) of the fused input norm (TMA kernel only, see fused_in_norm_ok)."""
        _dev(x)
        N, Hi, Wi, Ci_total = x.shape
        Ho, Wo = self.out_hw(Hi, Wi)
        dt = _dt(x)
        flags = extra_flags
        if stats is not None:
            flags |= CONV_STATS
        if in_stats is not None:
            flags |= CONV_IN_NORM
        if nchw_out is not None:
            flags |= CONV_OUT_NCHW_F32
            y, Co_total = nchw_out, self.Cout
        else:
            if out is None:
                out = torch.empty((N, Ho, Wo, self.Cout), device=x.device, dtype=x.dtype)
            y, Co_total = out, out.shape[3]
        if self.kind == "conv":
            d = make_desc(dt, N, Hi, Wi, Ci_total, ci_off, self.Cin, Ho, Wo, Co_total, co_off, self.Cout,
                          Ho, Wo, self.k, self.k, self.stride, self.pad, self.pad, self.dil, 1, 0, 0, act,
                          flags, in_act)
            conv_raw(d, x, wp, bias, y, stats, in_stats, in_affine)
        else:
            per_phase = self.Cout * 4 * self.Cin
            for ph in range(2):
                for pw in range(2):
                    d = make_desc(dt, N, Hi, Wi, Ci_total, ci_off, self.Cin, Ho, Wo, Co_total, co_off,
                                  self.Cout, Hi, Wi, 2, 2, 1, 1 - ph, 1 - pw, 1, 2, ph, pw, act, flags, in_act)
                    conv_raw(d, x, wp[(ph * 2 + pw) * per_phase:], bias, y, stats, in_stats, in_affine)
        return nchw_out if nchw_out is not None else out

    def dgrad(self, dy, wpd, in_hw, out=None, co_off=0, accumulate=False, dy_c_off=0):
        """dy: [N,Ho,Wo,Cdy_total] (the slice [dy_c_off, dy_c_off+Cout) is this conv's output grad).
        Returns / writes dx [N,Hi,Wi,*] channels [co_off, co_off+Cin)."""
        _dev(dy)
        N, Ho, Wo, Cdy = dy.shape
        Hi, Wi = in_hw
        dt = _dt(dy)
        if out is None:
            out = torch.empty((N, Hi, Wi, self.Cin), device=dy.device, dtype=dy.dtype)
        Co_total = out.shape[3]
        flags = CONV_ACCUM if accumulate else 0
        if self.kind == "convT":  # dgrad of convT = 4x4 s2 p1 conv over dy
            d = make_desc(dt, N, Ho, Wo, Cdy, dy_c_off, self.Cout, Hi, Wi, Co_total, co_off, self.Cin,
                          Hi, Wi, 4, 4, 2, 1, 1, 1, 1, 0, 0, ACT_NONE, flags)
            conv_raw(d, dy, wpd, None, out)
        elif self.stride == 2:  # dgrad of 4x4 s2 p1 conv = transposed conv phases over dy
            per_phase = self.Cin * 4 * self.Cout
            for ph in range(2):
                for pw in range(2):
                    d = make_desc(dt, N, Ho, Wo, Cdy, dy_c_off, self.Cout, Hi, Wi, Co_total, co_off,
                                  self.Cin, Ho, Wo, 2, 2, 1, 1 - ph, 1 - pw, 1, 2, ph, pw, ACT_NONE, flags)
                    conv_raw(d, dy, wpd[(ph * 2 + pw) * per_phase:], None, out)
        else:
            padp = self.dil * (self.k - 1) - self.pad
            d = make_desc(dt, N, Ho, Wo, Cdy, dy_c_off, self.Cout, Hi, Wi, Co_total, co_off, self.Cin,
                          Hi, Wi, self.k, self.k, 1, padp, padp, self.dil, 1, 0, 0, ACT_NONE, flags)
            conv_raw(d, dy, wpd, None, out)
        return out

    def wgrad(self, x, dy, dw, db=None, dy_c_off=0, ci_off=0, extra_flags=0, scratch=None):
        """Accumulates into dw (fp32, PyTorch weight layout) and db (fp32 [Cout]).  scratch: optional ZEROED fp32 buffer of
        dw.numel() elements for the packed gradient (a slice of the caller's arena instead of one allocation + memset per call)."""
        _dev(x)
        N, Hi, Wi, Ci_total = x.shape
        _, Ho, Wo, Cdy = dy.shape
        dt = _dt(x)
        dwp = scratch if scratch is not None else torch.zeros(dw.numel(), device=x.device, dtype=torch.float32)
        if self.kind == "conv":
            d = make_desc(dt, N, Hi, Wi, Ci_total, ci_off, self.Cin, Ho, Wo, Cdy, dy_c_off, self.Cout, Ho, Wo,
                          self.k, self.k, self.stride, self.pad, self.pad, self.dil, flags=extra_flags)
            _lib.call("msg_conv2d_wgrad", ctypes.byref(d), _p(x), _p(dy), _p(dwp), _stream())
            unpack_wgrad(dwp, dw.shape, PACK_FWD, dw)
        else:
            per_phase = self.Cout * 4 * self.Cin
            for ph in range(2):
                for pw in range(2):
                    d = make_desc(dt, N, Hi, Wi, Ci_total, ci_off, self.Cin, Ho, Wo, Cdy, dy_c_off, self.Cout,
                                  Hi, Wi, 2, 2, 1, 1 - ph, 1 - pw, 1, 2, ph, pw, flags=extra_flags)
                    _lib.call("msg_conv2d_wgrad", ctypes.byref(d), _p(x), _p(dy),
                              _p(dwp[(ph * 2 + pw) * per_phase:]), _stream())
            unpack_wgrad(dwp, dw.shape, PACK_CONVT_PHASES, dw)
        if db is not None:
            bias_grad(dy, db, dy_c_off, self.Cout)


def bias_grad(dy, db, c_off=0, C=None):
    N, H, W, Ct = dy.shape
    C = Ct if C is None else C
    if dy.dtype == torch.bfloat16 and C % 3 == 0 and C // 3 <= 256 and (C // 3) & (C // 3 - 1) == 0 and C // 3 >= 64:
        # the qkv convs (3C channels): three power-of-two slices on the vectorised kernel (0.011 ms each) instead of one launch
        # of the generic one (0.053 ms)
        part = C // 3
        for i in range(3):
            _lib.call("msg_bias_grad", _dt(dy), _p(dy), N * H * W, Ct, c_off + i * part, part, _p(db[i * part:]), _stream())
        return
    _lib.call("msg_bias_grad", _dt(dy), _p(dy), N * H * W, Ct, c_off, C, _p(db), _stream())


# ---- InstanceNorm -------------------------------------------------------------------------------
def new_stats(N, C, device):
    return torch.zeros((N, C, 2), device=device, dtype=torch.float64)


def instnorm_stats(x, stats=None):
    _dev(x)
    N, H, W, C = x.shape
    if stats is None:
        stats = new_stats(N, C, x.device)
    _lib.call("msg_instnorm_stats", _dt(x), _p(x), N, H * W, C, _p(stats), _stream())
    return stats


def instnorm_apply(x, stats, act=ACT_RELU, residual=None, out=None, gammas=None, betas=None, w=None, affine=None):
    """affine: (gamma, beta, img_stride) table (include/msg_b200.h) instead of the blend of gammas / betas by w."""
    _dev(x)
    N, H, W, C = x.shape
    if out is None:
        out = torch.empty_like(x)
    S = 0 if gammas is None else gammas.shape[0]
    if affine is None:
        _lib.call("msg_instnorm_apply", _dt(x), _p(x), _p(stats), N, H * W, C, act, _p(residual), S,
                  _p(gammas), _p(betas), _p(w), _p(out), _stream())
    else:
        _lib.call("msg_instnorm_apply_affine", _dt(x), _p(x), _p(stats), N, H * W, C, act, _p(residual), S,
                  _p(gammas), _p(betas), _p(w), *_aff(affine), _p(out), _stream())
    return out


def instnorm_bwd(x, stats, dy, act=ACT_RELU, out=None, return_scratch=False):
    """return_scratch: also return the kernel's per-(n, c) reductions [N, C, 2] = (sum g, sum g * xhat) with
    g = dy * act'(xhat) -- for a BatchNorm (N = 1 view) these are d(beta) and d(gamma)."""
    _dev(x)
    N, H, W, C = x.shape
    if out is None:
        out = torch.empty_like(x)
    scratch = torch.empty((N, C, 2), device=x.device, dtype=torch.float64)
    _lib.call("msg_instnorm_bwd", _dt(x), _p(x), _p(stats), _p(dy), N, H * W, C, act, _p(scratch), _p(out), _stream())
    return (out, scratch) if return_scratch else out


def _affine(gamma, beta, C):
    if (gamma is None) != (beta is None):
        raise _lib.MsgError("instnorm backward: gamma and beta go together")
    if gamma is not None and not (gamma.dtype == beta.dtype == torch.float32 and gamma.numel() == beta.numel() == C
                                  and gamma.is_contiguous() and beta.is_contiguous()):
        raise _lib.MsgError(f"instnorm backward: gamma / beta must be contiguous float32 [{C}]")


def instnorm_bwd_reduce(x, stats, dy, act=ACT_RELU, gamma=None, beta=None):
    """First half of instnorm_bwd: the fp64 per-(n, c) sums [N, C, 2] = (sum g, sum g * xhat), g = dy * act'(z) with
    z = xhat * gamma + beta (gamma / beta: optional fp32 [C]).  A synchronised BatchNorm all-reduces them (for a BatchNorm,
    N = 1 view, the local sums are d(beta) and d(gamma)) and rescales them to the local count before instnorm_bwd_apply."""
    _dev(x)
    N, H, W, C = x.shape
    _affine(gamma, beta, C)
    sums = torch.empty((N, C, 2), device=x.device, dtype=torch.float64)
    _lib.call("msg_instnorm_bwd_reduce", _dt(x), _p(x), _p(stats), _p(dy), N, H * W, C, act, _p(gamma), _p(beta), _p(sums),
              _stream())
    return sums


def instnorm_bwd_apply(x, stats, dy, sums, act=ACT_RELU, gamma=None, beta=None, out=None):
    """Second half of instnorm_bwd: dx = gamma * rstd * (g - sums[..., 0] / HW - xhat * sums[..., 1] / HW)."""
    _dev(x)
    N, H, W, C = x.shape
    _affine(gamma, beta, C)
    if out is None:
        out = torch.empty_like(x)
    _lib.call("msg_instnorm_bwd_apply", _dt(x), _p(x), _p(stats), _p(dy), N, H * W, C, act, _p(gamma), _p(beta), _p(sums),
              _p(out), _stream())
    return out


def instnorm_bwd_reduce_affine(x, stats, dy, affine, sums, act=ACT_RELU):
    """instnorm_bwd_reduce with a per-image affine (gamma, beta, img_stride): writes the (sum g, sum g * xhat) = (d beta_n,
    d gamma_n) of its C channels into `sums`, a flat fp64 view whose rows are img_stride channels apart (the layout of the
    affine tables)."""
    _dev(x)
    N, H, W, C = x.shape
    _lib.call("msg_instnorm_bwd_reduce_affine", _dt(x), _p(x), _p(stats), _p(dy), N, H * W, C, act, *_aff(affine), _p(sums),
              _stream())
    return sums


def instnorm_bwd_apply_affine(x, stats, dy, sums, affine, act=ACT_RELU, out=None):
    _dev(x)
    N, H, W, C = x.shape
    if out is None:
        out = torch.empty_like(x)
    _lib.call("msg_instnorm_bwd_apply_affine", _dt(x), _p(x), _p(stats), _p(dy), N, H * W, C, act, *_aff(affine), _p(sums),
              _p(out), _stream())
    return out


def style_affine(w, gammas, betas):
    """Per-image affine tables gamma / beta [N, Ct] = w [N, S] @ gammas / betas [S, Ct] (msg_style_affine: fmaf chain over s)."""
    _dev(w)
    N, S = w.shape
    Ct = gammas.shape[1]
    g = torch.empty((N, Ct), device=w.device, dtype=torch.float32)
    b = torch.empty_like(g)
    _lib.call("msg_style_affine", _p(w), N, S, _p(gammas), _p(betas), Ct, _p(g), _p(b), _stream())
    return g, b


def style_affine_bwd(sums, w, dgammas, dbetas):
    """dgammas / dbetas [S, Ct] += the gradients of style_affine's tables from one sums arena [N, Ct, 2] fp64."""
    N, S = w.shape
    _lib.call("msg_style_affine_bwd", _p(sums), _p(w), N, S, dgammas.shape[1], _p(dgammas), _p(dbetas), _stream())


# ---- LocalAttention core -------------------------------------------------------------------------
def local_attn_fwd(qkv, ws=4):
    _dev(qkv)
    N, H, W, C3 = qkv.shape
    C = C3 // 3
    out = torch.empty((N, H, W, C), device=qkv.device, dtype=qkv.dtype)
    _lib.call("msg_local_attn_fwd", _dt(qkv), _p(qkv), N, H, W, C, ws, _p(out), _stream())
    return out


def local_attn_bwd(qkv, dout, ws=4):
    N, H, W, C3 = qkv.shape
    dqkv = torch.empty_like(qkv)
    _lib.call("msg_local_attn_bwd", _dt(qkv), _p(qkv), _p(dout), N, H, W, C3 // 3, ws, _p(dqkv), _stream())
    return dqkv


def la_stage_supported(x, wqkv, wproj):
    """True when the fused LocalAttention stage kernel (csrc/la_stage.cu) takes this input: bf16, C in {64, 128}."""
    if x.dtype != torch.bfloat16 or not x.is_cuda:
        return False
    N, H, W, C = x.shape
    return _lib.load().msg_la_stage_supported(_dt(x), N, H, W, C, _p(x), _p(wqkv), _p(wproj), _p(x)) == 1


def la_stage_fwd(x, wqkv, bqkv, wproj, bproj, in_stats=None, in_act=ACT_NONE, out=None, in_affine=None):
    """LocalAttention.forward (enhanced_generator.py:13-47) in one launch: [IN + act of the producer] -> qkv 1x1 ->
    4x4-window channel attention -> proj 1x1.  x: [N,H,W,C] bf16 (raw conv output with `in_stats`, else normalised);
    wqkv / wproj: packed bf16 1x1 weights ([3C][C], [C][C]); biases fp32."""
    _dev(x)
    N, H, W, C = x.shape
    if out is None:
        out = torch.empty_like(x)
    if in_affine is None:
        _lib.call("msg_la_stage_fwd", _dt(x), _p(x), _p(in_stats), in_act, _p(wqkv), _p(bqkv), _p(wproj), _p(bproj), N, H, W, C,
                  _p(out), _stream())
    else:
        _lib.call("msg_la_stage_fwd_affine", _dt(x), _p(x), _p(in_stats), *_aff(in_affine), in_act, _p(wqkv), _p(bqkv), _p(wproj),
                  _p(bproj), N, H, W, C, _p(out), _stream())
    return out


# ---- layout / blend ------------------------------------------------------------------------------
def nchw_to_nhwc(x, dtype, Cp=None):
    _dev(x)
    x = x.detach()
    if x.dtype != torch.float32 or not x.is_contiguous():
        x = x.float().contiguous()
    N, C, H, W = x.shape
    Cp = C if Cp is None else Cp
    y = torch.empty((N, H, W, Cp), device=x.device, dtype=dtype)
    _lib.call("msg_nchw_to_nhwc", _DT[dtype], _p(x), N, C, H, W, Cp, _p(y), _stream())
    return y


def nhwc_to_nchw(x, C=None):
    _dev(x)
    N, H, W, Cp = x.shape
    C = Cp if C is None else C
    y = torch.empty((N, C, H, W), device=x.device, dtype=torch.float32)
    _lib.call("msg_nhwc_to_nchw", _dt(x), _p(x), N, C, H, W, Cp, _p(y), _stream())
    return y


def blend_outputs(ys, w, x=None, w_x=0.0, gain=1.0, clip=None, out_uint8=False, out=None):
    """out = gain * (sum_s w[s]*ys[s] + w_x*x), optional clip; optionally also the uint8 image
    ((v+1)/2 -> clamp -> *255).  ys: list of fp32 CUDA tensors of identical shape."""
    ys = [y.detach().contiguous() for y in ys]
    _dev(ys[0])
    S = len(ys)
    assert S == len(w)
    ptrs = (ctypes.c_void_p * S)(*[y.data_ptr() for y in ys])
    ws = (ctypes.c_float * S)(*[float(v) for v in w])
    if out is not None and out.dtype == torch.uint8:
        u8, out = out, None
        assert u8.is_contiguous() and u8.shape == ys[0].shape
    else:
        if out is None:
            out = torch.empty_like(ys[0])
        assert out.is_contiguous() and out.shape == ys[0].shape and out.dtype == torch.float32
        u8 = torch.empty(ys[0].shape, device=ys[0].device, dtype=torch.uint8) if out_uint8 else None
    lo, hi = (clip if clip is not None else (0.0, 0.0))
    xx = None if x is None else x.detach().contiguous()
    _lib.call("msg_blend_outputs", ptrs, ws, S, _p(xx), float(w_x), float(gain), int(clip is not None),
              float(lo), float(hi), ys[0].numel(), _p(out), _p(u8), _stream())
    if out is None:
        return u8
    return (out, u8) if out_uint8 else out


def blend_maps(ys, maps, x=None, gain=1.0, clip=None, normalize=False, out_uint8=False, out=None):
    """Per-pixel blend: out[n,:,i,j] = gain * (sum_k m_k(n,i,j) * plane_k[n,:,i,j]), optional clip / uint8 as blend_outputs.
    ys: S fp32 CUDA tensors [N,C,H,W]; maps: fp32 CUDA [Bm,K,h,w] with Bm in {1, N}, K in {S, S+1} (map S weights x),
    h <= H, w <= W, sampled bilinearly (align_corners=False) at each pixel; normalize divides the K weights by their sum."""
    ys = [y.detach().contiguous() for y in ys]
    _dev(ys[0])
    S = len(ys)
    N, C, H, W = ys[0].shape
    maps = maps.detach()
    assert maps.dtype == torch.float32 and maps.dim() == 4 and maps.is_contiguous(), "maps: contiguous fp32 [Bm,K,h,w]"
    _dev(maps)
    Bm, K, h, w = maps.shape
    ptrs = (ctypes.c_void_p * S)(*[y.data_ptr() for y in ys])
    if out is not None and out.dtype == torch.uint8:
        u8, out = out, None
        assert u8.is_contiguous() and u8.shape == ys[0].shape
    else:
        if out is None:
            out = torch.empty_like(ys[0])
        assert out.is_contiguous() and out.shape == ys[0].shape and out.dtype == torch.float32
        u8 = torch.empty(ys[0].shape, device=ys[0].device, dtype=torch.uint8) if out_uint8 else None
    lo, hi = (clip if clip is not None else (0.0, 0.0))
    xx = None if x is None else x.detach().contiguous()
    _lib.call("msg_blend_maps", ptrs, S, _p(xx), _p(maps), Bm, K, h, w, N, C, H, W, int(bool(normalize)), float(gain),
              int(clip is not None), float(lo), float(hi), _p(out), _p(u8), _stream())
    if out is None:
        return u8
    return (out, u8) if out_uint8 else out


def gaussian_blur(planes, sigma):
    """scipy.ndimage.gaussian_filter(mode="reflect", truncate=4.0) of every trailing [h, w] plane of an fp32 CUDA tensor."""
    _dev(planes)
    assert planes.dtype == torch.float32 and planes.dim() >= 2
    src = planes.detach().contiguous()
    h, w = src.shape[-2:]
    tmp = torch.empty_like(src)
    out = torch.empty_like(src)
    _lib.call("msg_gaussian_blur", _p(src), src.numel() // max(h * w, 1), h, w, float(sigma), _p(tmp), _p(out), _stream())
    return out


# ---- misc ----------------------------------------------------------------------------------------
def tanh_bwd_nchw(y, dy, dtype, Cp):
    N, C, H, W = y.shape
    dz = torch.empty((N, H, W, Cp), device=y.device, dtype=dtype)
    _lib.call("msg_tanh_bwd_nchw", _DT[dtype], _p(y), _p(dy.contiguous()), N, C, H, W, Cp, _p(dz), _stream())
    return dz


def act_bwd(y, dy, act):
    dx = torch.empty_like(y)
    _lib.call("msg_act_bwd", _dt(y), _p(y), _p(dy), y.numel(), act, _p(dx), _stream())
    return dx


def add(a, b, out=None):
    if out is None:
        out = torch.empty_like(a)
    _lib.call("msg_add", _dt(a), _p(a), _p(b), a.numel(), _p(out), _stream())
    return out


def avgpool_fwd(x):
    N, H, W, C = x.shape
    y = torch.empty((N, C), device=x.device, dtype=torch.float32)
    _lib.call("msg_avgpool_fwd", _dt(x), _p(x), N, H * W, C, _p(y), _stream())
    return y


def avgpool_bwd(dy, shape, dtype):
    N, H, W, C = shape
    dx = torch.empty(shape, device=dy.device, dtype=dtype)
    _lib.call("msg_avgpool_bwd", _DT[dtype], _p(dy.contiguous()), N, H * W, C, _p(dx), _stream())
    return dx


def maxpool_fwd(x):
    N, H, W, C = x.shape
    y = torch.empty((N, H // 2, W // 2, C), device=x.device, dtype=x.dtype)
    _lib.call("msg_maxpool2x2_fwd", _dt(x), _p(x), N, H, W, C, _p(y), _stream())
    return y


def maxpool_bwd(x, dy):
    N, H, W, C = x.shape
    dx = torch.empty_like(x)
    _lib.call("msg_maxpool2x2_bwd", _dt(x), _p(x), _p(dy), N, H, W, C, _p(dx), _stream())
    return dx


def mse_loss(a, b=None, b_const=0.0, scale=1.0, want_grad=True):
    """Returns (loss [1] fp32 device tensor, grad_a or None).  a: fp32 tensor."""
    a = a.contiguous()
    loss = torch.zeros(1, device=a.device, dtype=torch.float32)
    ga = torch.empty_like(a) if want_grad else None
    _lib.call("msg_mse_loss", _p(a), _p(b), float(b_const), a.numel(), float(scale), _p(loss), _p(ga), _stream())
    return loss, ga


def l1_loss(a, b=None, b_const=0.0, scale=1.0, want_grad_a=True, want_grad_b=False):
    a = a.contiguous()
    loss = torch.zeros(1, device=a.device, dtype=torch.float32)
    ga = torch.empty_like(a) if want_grad_a else None
    gb = torch.empty_like(a) if want_grad_b else None
    _lib.call("msg_l1_loss", _p(a), _p(b), float(b_const), a.numel(), float(scale), _p(loss), _p(ga), _p(gb), _stream())
    return loss, ga, gb


def adam_step(p, g, m, v, lr, beta1, beta2, eps, step, grad_scale=1.0):
    _lib.call("msg_adam_step", _p(p), _p(g), _p(m), _p(v), p.numel(), float(lr), float(beta1), float(beta2),
              float(eps), int(step), float(grad_scale), _stream())


def u8_canvas_to_nchw(img_u8, H=None, W=None, off_y=0, off_x=0, fill=255, want_canvas=False):
    """uint8 [N,h,w,3] (PIL layout, on the device) -> fp32 NCHW [N,3,H,W] normalised to [-1,1] after pasting on an HxW canvas
    (batch_process_images.py:193-205); with want_canvas also the uint8 canvas [N,H,W,3]."""
    _dev(img_u8)
    assert img_u8.dtype == torch.uint8 and img_u8.dim() == 4 and img_u8.shape[3] == 3 and img_u8.is_contiguous()
    N, h, w, _ = img_u8.shape
    H, W = (h if H is None else H), (w if W is None else W)
    out = torch.empty((N, 3, H, W), device=img_u8.device, dtype=torch.float32)
    canvas = torch.empty((N, H, W, 3), device=img_u8.device, dtype=torch.uint8) if want_canvas else None
    _lib.call("msg_u8_canvas_to_nchw", _p(img_u8), N, h, w, H, W, int(off_y), int(off_x), int(fill), _p(out), _p(canvas), _stream())
    return (out, canvas) if want_canvas else out


def u8_strength_blend(orig_nhwc, styled_nchw, strength):
    """uint8(clip(orig * (1 - s) + styled * s, 0, 255)) (batch_process_images.py:304-310); orig NHWC, styled NCHW -> NHWC."""
    _dev(orig_nhwc)
    N, H, W, _ = orig_nhwc.shape
    assert orig_nhwc.dtype == styled_nchw.dtype == torch.uint8 and tuple(styled_nchw.shape) == (N, 3, H, W)
    out = torch.empty_like(orig_nhwc)
    _lib.call("msg_u8_strength_blend", _p(orig_nhwc.contiguous()), _p(styled_nchw.contiguous()), N, H, W, float(strength), _p(out), _stream())
    return out


def adam_step_dev(p, g, m, v, lr, beta1, beta2, eps, step_dev, grad_scale=1.0):
    """as adam_step with the step count in device memory (int32 tensor, incremented by the call): graph-replayable"""
    _lib.call("msg_adam_step_dev", _p(p), _p(g), _p(m), _p(v), p.numel(), float(lr), float(beta1), float(beta2),
              float(eps), _p(step_dev), float(grad_scale), _stream())


def spectral_norm(w2d_like, rows, cols, u, v, do_iter, sigma, eps=1e-12):
    _lib.call("msg_spectral_norm", _p(w2d_like), rows, cols, _p(u), _p(v), int(do_iter), float(eps), _p(sigma), _stream())


def spectral_norm_batched(problems, do_iter, eps=1e-12):
    """problems: [(w2d_like, rows, cols, u, v, sigma[1])], at most 8: one launch for all of them (csrc/elementwise.cu)"""
    b = _lib.SnBatch()
    b.n = len(problems)
    for i, (w, rows, cols, u, v, sigma) in enumerate(problems):
        b.w[i], b.u[i], b.v[i], b.sigma[i], b.rows[i], b.cols[i] = w.data_ptr(), u.data_ptr(), v.data_ptr(), sigma.data_ptr(), rows, cols
    _lib.call("msg_spectral_norm_batched", ctypes.byref(b), int(do_iter), float(eps), _stream())


def spectral_norm_bwd(dw, w_orig, u, v, sigma, rows, cols, dw_orig):
    scratch = torch.empty(1, device=dw.device, dtype=torch.float32)
    _lib.call("msg_spectral_norm_bwd", _p(dw), _p(w_orig), _p(u), _p(v), _p(sigma), rows, cols, _p(dw_orig), _p(scratch), _stream())


def gram(feat):
    N, H, W, C = feat.shape
    g = torch.empty((N, C, C), device=feat.device, dtype=torch.float32)
    _lib.call("msg_gram", _dt(feat), _p(feat), N, H * W, C, _p(g), _stream())
    return g


def gram_loss_fwd(feat, target, scale=1.0, loss=None):
    N, H, W, C = feat.shape
    g = torch.empty((N, C, C), device=feat.device, dtype=torch.float32)
    if loss is None:
        loss = torch.zeros(1, device=feat.device, dtype=torch.float32)
    _lib.call("msg_gram_loss_fwd", _dt(feat), _p(feat), N, H * W, C, _p(target), float(scale), _p(g), _p(loss), _stream())
    return loss, g


def gram_loss_bwd(feat, g, target, scale=1.0):
    N, H, W, C = feat.shape
    dfeat = torch.empty_like(feat)
    wscratch = torch.empty((N, C, C), device=feat.device, dtype=feat.dtype)
    _lib.call("msg_gram_loss_bwd", _dt(feat), _p(feat), N, H * W, C, _p(g), _p(target), float(scale),
              _p(wscratch), _p(dfeat), _stream())
    return dfeat
