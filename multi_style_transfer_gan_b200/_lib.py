"""ctypes binding of libmsg_b200.so (the C-ABI declared in include/msg_b200.h).

There is no CPU or PyTorch fallback: if the shared library is missing, or the device is not a
B200 (sm_100), every op raises.  Build with ``python -m multi_style_transfer_gan_b200.build``.
"""
import ctypes
import os
import threading

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("MSG_B200_LIB") or os.path.join(HERE, "libmsg_b200.so")   # (env: development A/B builds)

F32, BF16 = 0, 1
ACT_NONE, ACT_RELU, ACT_LRELU, ACT_TANH = 0, 1, 2, 3
CONV_STATS, CONV_OUT_NCHW_F32, CONV_IN_NORM, CONV_ACCUM, CONV_FORCE_SIMT, CONV_FORCE_GATHER = 1, 2, 4, 8, 256, 512
CONV_PER_IMAGE_W = 16
PACK_FWD, PACK_DGRAD_S1, PACK_CONVT_PHASES = 0, 1, 2

c_int, c_ll, c_float, c_void_p, c_uint = (ctypes.c_int, ctypes.c_longlong, ctypes.c_float,
                                          ctypes.c_void_p, ctypes.c_uint)


class ConvDesc(ctypes.Structure):
    _fields_ = [(n, c_int) for n in (
        "dtype", "N", "Hi", "Wi", "Ci_total", "ci_off", "Cin", "Ho", "Wo", "Co_total", "co_off",
        "Cout", "Hg", "Wg", "KH", "KW", "in_stride", "pad_h", "pad_w", "dil", "out_stride",
        "out_off_h", "out_off_w", "act")] + [("flags", c_uint), ("in_act", c_int)]


SLAB_MAX_KBLOCKS, SLAB_MAX_TAPS = 32, 128


class SlabDesc(ctypes.Structure):
    """mirrors msg_slab_desc (include/msg_b200.h)"""
    _fields_ = [(n, c_int) for n in (
        "dtype", "N", "H", "W", "Ci_total", "ci_off", "Cin", "Co_total", "co_off", "out_stride", "out_off_h", "out_off_w", "Ntot", "n_store", "ncols",
        "halo", "pixel_pair_k", "n_chains", "act")] + [("flags", c_uint), ("n_kblocks", c_int), ("n_taps", c_int),
        ("kb_dy", c_int * SLAB_MAX_KBLOCKS), ("kb_cb", c_int * SLAB_MAX_KBLOCKS),
        ("kb_tap_begin", c_int * (SLAB_MAX_KBLOCKS + 1)),
        ("tap_sx", c_int * SLAB_MAX_TAPS), ("tap_acc_col", c_int * SLAB_MAX_TAPS),
        ("tap_first", c_int * SLAB_MAX_TAPS), ("tap_kstep", c_int * SLAB_MAX_TAPS)]


SHIFT_MAX_KBLOCKS, SHIFT_MAX_GROUPS, SHIFT_MAX_TERMS = 32, 8, 32


class ShiftDesc(ctypes.Structure):
    """mirrors msg_shift_desc (include/msg_b200.h)"""
    _fields_ = [(n, c_int) for n in (
        "dtype", "N", "H", "W", "Ci_total", "ci_off", "Cin", "Co_total", "co_off", "Ntot", "n_out", "halo", "act")] + [
        ("flags", c_uint), ("n_kblocks", c_int), ("n_groups", c_int), ("n_terms", c_int)] + [
        (n, c_int * SHIFT_MAX_KBLOCKS) for n in ("kb_dy", "kb_cb", "kb_col0", "kb_ncols", "kb_wrow", "kb_first")] + [
        (n, c_int * SHIFT_MAX_GROUPS) for n in ("grp_col0", "grp_span", "grp_out_col0", "grp_out_cols")] + [
        ("grp_term_begin", c_int * (SHIFT_MAX_GROUPS + 1)),
        ("term_shift", c_int * SHIFT_MAX_TERMS), ("term_col", c_int * SHIFT_MAX_TERMS),
        ("tile_rows", c_int), ("kb_same_slab", c_int * SHIFT_MAX_KBLOCKS), ("grp_row", c_int * SHIFT_MAX_GROUPS)]


class MsbRingDesc(ctypes.Structure):
    """mirrors msg_msb_ring_desc (include/msg_b200.h)"""
    _fields_ = [(n, c_int) for n in ("dtype", "N", "H", "W", "Ci_total", "ci_off", "Co_total", "co_off")] + [("flags", c_uint)]


class ConvtRingDesc(ctypes.Structure):
    """mirrors msg_convt_ring_desc (include/msg_b200.h)"""
    _fields_ = [(n, c_int) for n in ("dtype", "N", "H", "W", "Cin", "Cout", "Ci_total", "ci_off", "Co_total", "co_off")] + [("flags", c_uint)]


class Out7RingDesc(ctypes.Structure):
    """mirrors msg_out7_ring_desc (include/msg_b200.h)"""
    _fields_ = [(n, c_int) for n in ("dtype", "N", "H", "W", "Cf_total", "cf_off", "Cr_total", "cr_off", "Cs_total", "cs_off")]


class DownRingDesc(ctypes.Structure):
    """mirrors msg_down_ring_desc (include/msg_b200.h)"""
    _fields_ = [(n, c_int) for n in ("dtype", "N", "H", "W", "Cout", "Ci_total", "ci_off", "Co_total", "co_off", "Cs_total", "cs_off")] + [("flags", c_uint)]


SN_MAX_BATCH = 8


class SnBatch(ctypes.Structure):
    """mirrors msg_sn_batch (include/msg_b200.h)"""
    _fields_ = [("w", c_void_p * SN_MAX_BATCH), ("u", c_void_p * SN_MAX_BATCH), ("v", c_void_p * SN_MAX_BATCH),
                ("sigma", c_void_p * SN_MAX_BATCH), ("rows", c_int * SN_MAX_BATCH), ("cols", c_int * SN_MAX_BATCH), ("n", c_int)]


_P = c_void_p
# name -> argtypes (everything returns int except msg_last_error)
SIGNATURES = {
    "msg_version": [],
    "msg_check_device": [],
    "msg_sm_count": [],
    "msg_conv2d": [ctypes.POINTER(ConvDesc), _P, _P, _P, _P, _P, _P, _P],
    "msg_conv2d_path": [ctypes.POINTER(ConvDesc), _P, _P, _P],
    "msg_conv2d_affine": [ctypes.POINTER(ConvDesc), _P, _P, _P, _P, _P, _P, _P, _P, c_int, _P],
    "msg_style_affine": [_P, c_int, c_int, _P, _P, c_int, _P, _P, _P],
    "msg_style_affine_bwd": [_P, _P, c_int, c_int, c_int, _P, _P, _P],
    "msg_conv2d_wgrad": [ctypes.POINTER(ConvDesc), _P, _P, _P, _P],
    "msg_conv_slab": [ctypes.POINTER(SlabDesc), _P, _P, _P, _P, _P, _P],
    "msg_conv_shift": [ctypes.POINTER(ShiftDesc), _P, _P, _P, _P, _P, _P],
    "msg_pack_conv_weight": [_P, c_int, c_int, c_int, c_int, c_int, c_int, _P, _P, _P],
    "msg_unpack_conv_wgrad": [_P, c_int, c_int, c_int, c_int, c_int, _P, _P],
    "msg_bias_grad": [c_int, _P, c_ll, c_int, c_int, c_int, _P, _P],
    "msg_instnorm_stats": [c_int, _P, c_int, c_ll, c_int, _P, _P],
    "msg_instnorm_apply": [c_int, _P, _P, c_int, c_ll, c_int, c_int, _P, c_int, _P, _P, _P, _P, _P],
    "msg_instnorm_bwd": [c_int, _P, _P, _P, c_int, c_ll, c_int, c_int, _P, _P, _P],
    "msg_instnorm_bwd_reduce": [c_int, _P, _P, _P, c_int, c_ll, c_int, c_int, _P, _P, _P, _P],
    "msg_instnorm_bwd_apply": [c_int, _P, _P, _P, c_int, c_ll, c_int, c_int, _P, _P, _P, _P, _P],
    "msg_instnorm_apply_affine": [c_int, _P, _P, c_int, c_ll, c_int, c_int, _P, c_int, _P, _P, _P, _P, _P, c_int, _P, _P],
    "msg_instnorm_bwd_reduce_affine": [c_int, _P, _P, _P, c_int, c_ll, c_int, c_int, _P, _P, c_int, _P, _P],
    "msg_instnorm_bwd_apply_affine": [c_int, _P, _P, _P, c_int, c_ll, c_int, c_int, _P, _P, c_int, _P, _P, _P],
    "msg_local_attn_fwd": [c_int, _P, c_int, c_int, c_int, c_int, c_int, _P, _P],
    "msg_local_attn_bwd": [c_int, _P, _P, c_int, c_int, c_int, c_int, c_int, _P, _P],
    "msg_la_stage_set_trace": [_P],
    "msg_la_stage_supported": [c_int, c_int, c_int, c_int, c_int, _P, _P, _P, _P],
    "msg_la_stage_fwd": [c_int, _P, _P, c_int, _P, _P, _P, _P, c_int, c_int, c_int, c_int, _P, _P],
    "msg_la_stage_fwd_affine": [c_int, _P, _P, _P, _P, c_int, c_int, _P, _P, _P, _P, c_int, c_int, c_int, c_int, _P, _P],
    "msg_nchw_to_nhwc": [c_int, _P, c_int, c_int, c_int, c_int, c_int, _P, _P],
    "msg_nhwc_to_nchw": [c_int, _P, c_int, c_int, c_int, c_int, c_int, _P, _P],
    "msg_blend_outputs": [ctypes.POINTER(_P), ctypes.POINTER(c_float), c_int, _P, c_float, c_float,
                          c_int, c_float, c_float, c_ll, _P, _P, _P],
    "msg_blend_maps": [ctypes.POINTER(_P), c_int, _P, _P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int,
                       c_float, c_int, c_float, c_float, _P, _P, _P],
    "msg_gaussian_blur": [_P, c_ll, c_int, c_int, c_float, _P, _P, _P],
    "msg_mse_loss": [_P, _P, c_float, c_ll, c_float, _P, _P, _P],
    "msg_l1_loss": [_P, _P, c_float, c_ll, c_float, _P, _P, _P, _P],
    "msg_msb64_ring": [ctypes.POINTER(MsbRingDesc), _P, _P, _P, _P, _P, _P],
    "msg_msb_ring": [ctypes.POINTER(MsbRingDesc), ctypes.c_int, _P, _P, _P, _P, _P, _P],
    "msg_convt_ring": [ctypes.POINTER(ConvtRingDesc), _P, _P, _P, _P, _P, _P],
    "msg_out7_ring": [ctypes.POINTER(Out7RingDesc), _P, _P, _P, _P, _P, _P, _P],
    "msg_down_ring": [ctypes.POINTER(DownRingDesc), _P, _P, _P, _P, _P, _P, _P],
    "msg_out7_ring_affine": [ctypes.POINTER(Out7RingDesc), _P, _P, _P, _P, c_int, _P, _P, _P, _P, _P],
    "msg_down_ring_affine": [ctypes.POINTER(DownRingDesc), _P, _P, _P, _P, c_int, _P, _P, _P, _P, _P],
    "msg_u8_canvas_to_nchw": [_P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, _P, _P, _P],
    "msg_u8_strength_blend": [_P, _P, c_int, c_int, c_int, ctypes.c_double, _P, _P],
    "msg_adam_step": [_P, _P, _P, _P, c_ll, c_float, c_float, c_float, c_float, c_int, c_float, _P],
    "msg_adam_step_dev": [_P, _P, _P, _P, c_ll, c_float, c_float, c_float, c_float, _P, c_float, _P],
    "msg_spectral_norm": [_P, c_int, c_int, _P, _P, c_int, c_float, _P, _P],
    "msg_spectral_norm_batched": [ctypes.POINTER(SnBatch), c_int, c_float, _P],
    "msg_spectral_norm_bwd": [_P, _P, _P, _P, _P, c_int, c_int, _P, _P, _P],
    "msg_gram": [c_int, _P, c_int, c_ll, c_int, _P, _P],
    "msg_gram_loss_fwd": [c_int, _P, c_int, c_ll, c_int, _P, c_float, _P, _P, _P],
    "msg_gram_loss_bwd": [c_int, _P, c_int, c_ll, c_int, _P, _P, c_float, _P, _P, _P],
    "msg_maxpool2x2_fwd": [c_int, _P, c_int, c_int, c_int, c_int, _P, _P],
    "msg_maxpool2x2_bwd": [c_int, _P, _P, c_int, c_int, c_int, c_int, _P, _P],
    "msg_act_bwd": [c_int, _P, _P, c_ll, c_int, _P, _P],
    "msg_tanh_bwd_nchw": [c_int, _P, _P, c_int, c_int, c_int, c_int, c_int, _P, _P],
    "msg_add": [c_int, _P, _P, c_ll, _P, _P],
    "msg_avgpool_fwd": [c_int, _P, c_int, c_ll, c_int, _P, _P],
    "msg_avgpool_bwd": [c_int, _P, c_int, c_ll, c_int, _P, _P],
}

_lib = None
_lock = threading.Lock()
_device_ok = set()


class MsgError(RuntimeError):
    pass


def load():
    """Loads the shared library once; raises MsgError (never falls back) if it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise MsgError(
                f"{LIB_PATH} not found: the CUDA extension is not built and there is no fallback path. "
                "Run `python -m multi_style_transfer_gan_b200.build` (needs nvcc).")
        lib = ctypes.CDLL(LIB_PATH)
        for name, args in SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError if the .so is stale: loud on purpose
            fn.argtypes = args
            fn.restype = c_int
        lib.msg_last_error.argtypes = []
        lib.msg_last_error.restype = ctypes.c_char_p
        _lib = lib
    return _lib


def check(rc):
    if rc != 0:
        msg = load().msg_last_error()
        raise MsgError(f"msg_b200 error {rc}: {msg.decode(errors='replace') if msg else ''}")


def require_device(index):
    """Raises unless CUDA device `index` (the device that owns the tensors of the call) is sm_100; checked once per
    device.  msg_check_device() answers for the CURRENT device, so it is only consulted when that is `index`."""
    if index in _device_ok:
        return
    lib = load()
    import torch
    major, minor = torch.cuda.get_device_capability(index)
    if major != 10:
        raise MsgError(f"msg_b200 kernels are built for sm_100a only; cuda:{index} is sm_{major}{minor} (no fallback)")
    if torch.cuda.current_device() == index:
        check(lib.msg_check_device())
    _device_ok.add(index)


# launch counter: every successful C-ABI call that launches kernels bumps this (bench.py's
# gpu_launches claim is derived from it).
launches = 0
prof_hook = None   # set by profiler.start(): name -> end event to record after the launch


def call(name, *args):
    global launches
    end = prof_hook(name) if prof_hook is not None else None
    rc = getattr(load(), name)(*args)
    if end is not None:
        end.record()
    if rc != 0:
        check(rc)
    launches += 1
