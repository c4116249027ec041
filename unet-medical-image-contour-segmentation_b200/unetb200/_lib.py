"""ctypes binding of libunetb200.so (the C ABI declared in include/unetb200.h).

The library is built in-tree by ``make -C csrc`` (or ``__graft_entry__.build()``) and loaded from
this directory.  There is no fallback: if the shared object is missing or a call fails, the
caller gets an exception -- never a silent PyTorch/CPU path.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libunetb200.so")

F32, BF16, I64, U8 = 0, 1, 2, 3
ALGO_AUTO, ALGO_SIMT, ALGO_TC, ALGO_PREFER_TC = 0, 1, 2, 3
E_INVALID, E_CUDA, E_NOMEM = -1, -2, -3

c_i64 = C.c_int64
c_p = C.c_void_p


class GConv(C.Structure):
    """Mirror of unetb200_gconv_t."""
    _fields_ = [
        ("dtype", C.c_int32), ("algo", C.c_int32),
        ("B", C.c_int32), ("Hm", C.c_int32), ("Wm", C.c_int32),
        ("Cin", C.c_int32), ("ntaps", C.c_int32),
        ("tap_dy", C.c_int32 * 9), ("tap_dx", C.c_int32 * 9),
        ("in_scale", C.c_int32), ("in_off_y", C.c_int32), ("in_off_x", C.c_int32),
        ("Hin", C.c_int32), ("Win", C.c_int32), ("ld_in", c_i64),
        ("N", C.c_int32), ("nquad", C.c_int32), ("out_scale", C.c_int32),
        ("out_off_y", C.c_int32), ("out_off_x", C.c_int32),
        ("Hout", C.c_int32), ("Wout", C.c_int32), ("ld_out", c_i64),
    ]


class PackJob(C.Structure):
    """Mirror of unetb200_pack_job_t."""
    _fields_ = [("src", c_p), ("dst", c_p), ("n0", c_i64), ("n1", c_i64), ("n2", c_i64),
                ("s0", c_i64), ("s1", c_i64), ("s2", c_i64), ("off", c_i64)]


class ReduceJob(C.Structure):
    """Mirror of unetb200_reduce_job_t."""
    _fields_ = [("partials", c_p), ("dst", c_p), ("st", c_i64), ("sc", c_i64), ("sq", c_i64), ("sn", c_i64),
                ("splits", C.c_int32), ("ntaps", C.c_int32), ("Cin", C.c_int32), ("N", C.c_int32), ("Cq", C.c_int32),
                ("accumulate", C.c_int32)]


# name -> (restype, argtypes); every symbol include/unetb200.h declares
PROTOTYPES = {
    "unetb200_version": (C.c_int, []),
    "unetb200_last_error": (C.c_char_p, []),
    "unetb200_device_info": (C.c_int, [C.POINTER(C.c_int)] * 3),
    "unetb200_gconv_stats_workspace": (c_i64, [C.POINTER(GConv)]),
    "unetb200_gconv_fprop": (C.c_int, [C.POINTER(GConv), c_p, c_p, c_p, c_p, c_p, c_p, C.POINTER(C.c_int), c_p]),
    "unetb200_gconv_fprop_affine_relu_supported": (C.c_int, [C.POINTER(GConv), c_p, c_p, c_p]),
    "unetb200_gconv_fprop_affine_relu": (C.c_int, [C.POINTER(GConv), c_p, c_p, c_p, c_p, c_p]),
    "unetb200_gconv_fprop_affine_relu_pool_supported": (C.c_int, [C.POINTER(GConv), c_p, c_p, c_p, c_p, C.c_int64]),
    "unetb200_gconv_fprop_affine_relu_pool": (C.c_int, [C.POINTER(GConv), c_p, c_p, c_p, c_p, c_p, C.c_int64, c_p]),
    "unetb200_gconv_fprop_affine_relu_outconv_supported": (C.c_int, [C.POINTER(GConv), c_p, c_p, C.c_int]),
    "unetb200_gconv_fprop_affine_relu_outconv": (C.c_int, [C.POINTER(GConv), c_p, c_p, c_p, c_p, c_p, c_p, C.c_int, c_p]),
    "unetb200_wgrad_reduce_multi": (C.c_int, [C.POINTER(ReduceJob), C.c_int, c_p]),
    "unetb200_gconv_dgrad_bnbwd_supported": (C.c_int, [C.POINTER(GConv), c_p, c_p, c_p]),
    "unetb200_gconv_dgrad_bnbwd": (C.c_int, [C.POINTER(GConv), c_p, c_p, c_p, c_p, C.c_int64, c_p, c_p, c_p, c_p]),
    "unetb200_gconv_wgrad_plan": (C.c_int, [C.POINTER(GConv), C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "unetb200_gconv_wgrad": (C.c_int, [C.POINTER(GConv), c_p, c_p, c_p, C.c_int, c_p]),
    "unetb200_wgrad_reduce": (C.c_int, [c_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, c_p, c_i64, c_i64, c_i64, c_i64,
                                        C.c_int, c_p]),
    "unetb200_pack_weights": (C.c_int, [c_p, c_p, C.c_int, c_i64, c_i64, c_i64, c_i64, c_i64, c_i64, c_i64, c_p]),
    "unetb200_pack_weights_multi": (C.c_int, [C.POINTER(PackJob), C.c_int, C.c_int, c_p]),
    "unetb200_split_tf32": (C.c_int, [c_p, c_i64, c_p, c_i64, C.c_int, C.c_int, c_p]),
    "unetb200_bn_finalize": (C.c_int, [c_p, c_i64, c_p, c_p, C.c_float, C.c_float, c_p, c_p, c_p, c_p, c_p, c_p, C.c_int, c_p]),
    "unetb200_bn_finalize_track": (C.c_int, [c_p, c_i64, c_p, c_p, C.c_float, C.c_float, c_p, c_p, c_p, c_p, c_p, c_p, c_p,
                                             C.c_int, c_p]),
    "unetb200_bn_eval_coeffs": (C.c_int, [c_p, c_p, c_p, c_p, C.c_float, c_p, c_p, c_p, c_p, C.c_int, c_p]),
    "unetb200_bn_relu_apply": (C.c_int, [c_p, c_i64, c_p, c_p, c_p, c_i64, c_p, c_i64, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, c_p]),
    "unetb200_maxpool2_fwd": (C.c_int, [c_p, c_i64, c_p, c_i64, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, c_p]),
    "unetb200_maxpool2_bwd": (C.c_int, [c_p, c_i64, c_p, c_i64, c_p, c_i64, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, c_p]),
    "unetb200_bn_relu_bwd_reduce": (C.c_int, [c_p, c_i64, c_p, c_i64, c_p, c_p, c_p, c_p, c_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, c_p]),
    "unetb200_bn_bwd_finalize": (C.c_int, [c_p, c_i64, C.c_int, c_p, c_p, c_p, C.c_int, c_p]),
    "unetb200_bn_relu_bwd_apply": (C.c_int, [c_p, c_i64, c_p, c_i64, c_p, c_p, c_p, c_p, c_p, c_p, c_i64, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, c_p]),
    "unetb200_bn_peer_group_create": (C.c_int, [C.c_int, C.c_int, C.c_int, c_p, c_p, C.POINTER(c_p)]),
    "unetb200_bn_peer_group_open": (C.c_int, [c_p, c_p, c_p]),
    "unetb200_bn_peer_group_destroy": (C.c_int, [c_p]),
    "unetb200_bn_peer_group_status": (C.c_int, [c_p, C.POINTER(c_i64), C.POINTER(c_i64)]),
    "unetb200_bn_sync_finalize": (C.c_int, [c_p, c_p, c_i64, c_p, c_p, C.c_float, C.c_float, c_p, c_p, c_p, c_p, c_p, c_p,
                                            c_p, C.c_int, c_p]),
    "unetb200_bn_sync_bwd_finalize": (C.c_int, [c_p, c_p, c_i64, c_p, c_p, c_p, C.c_int, c_p]),
    "unetb200_upsample2x_fwd": (C.c_int, [c_p, c_i64, c_p, c_i64, C.c_int] + [C.c_int] * 8 + [c_p]),
    "unetb200_upsample2x_bwd": (C.c_int, [c_p, c_i64, c_p, c_i64, C.c_int] + [C.c_int] * 8 + [c_p]),
    "unetb200_gather_nhwc": (C.c_int, [c_p, C.c_int, c_i64, c_i64, c_i64, c_i64, c_p, C.c_int, c_i64, C.c_int, C.c_int, C.c_int, C.c_int, c_p]),
    "unetb200_copy_channels": (C.c_int, [c_p, C.c_int, c_i64, c_p, C.c_int, c_i64, c_i64, C.c_int, c_p]),
    "unetb200_zero_channels": (C.c_int, [c_p, C.c_int, c_i64, c_i64, C.c_int, c_p]),
    "unetb200_sa_forward": (C.c_int, [c_p, c_i64, c_p, c_p, c_p, c_p, c_i64, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, c_p]),
    "unetb200_sa_backward_workspace": (c_i64, [C.c_int, C.c_int, C.c_int]),
    "unetb200_sa_backward": (C.c_int, [c_p, c_i64, c_p, c_i64, c_p, c_p, c_p, c_p, c_i64, c_p, c_p, C.c_int, C.c_int, C.c_int,
                                       C.c_int, C.c_int, c_p]),
    "unetb200_maxpool2_bwd_bnreduce": (C.c_int, [c_p, c_i64, c_p, c_i64, c_p, c_i64, c_p, c_i64, c_p, c_p, c_p, c_p, c_p,
                                                 C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, c_p]),
    "unetb200_f64_to_f32": (C.c_int, [c_p, c_p, C.c_int, c_p]),
    "unetb200_channel_sum": (C.c_int, [c_p, C.c_int, c_i64, c_i64, C.c_int, c_p, c_p, c_p]),
    "unetb200_add_channels": (C.c_int, [c_p, c_i64, c_p, c_i64, C.c_int, c_i64, C.c_int, c_p]),
    "unetb200_outconv_fwd": (C.c_int, [c_p, c_i64, c_p, c_p, c_p, C.c_int, c_i64, C.c_int, C.c_int, c_p]),
    "unetb200_outconv_bwd_workspace": (c_i64, [c_i64, C.c_int, C.c_int]),
    "unetb200_outconv_bwd": (C.c_int, [c_p, c_i64, c_p, c_p, c_p, c_i64, c_p, c_p, c_p, C.c_int, c_i64, C.c_int, C.c_int, c_p]),
    "unetb200_outconv_bwd_bnbwd_supported": (C.c_int, [c_p, c_i64, c_p, c_i64, c_p, c_i64, C.c_int, C.c_int, C.c_int]),
    "unetb200_outconv_bwd_bnbwd": (C.c_int, [c_p, c_i64, c_p, c_p, c_p, c_i64, c_p, c_p, c_p, c_p, c_i64, c_p, c_p, C.c_int,
                                             c_i64, C.c_int, C.c_int, c_p]),
    "unetb200_ce_dice_fwd": (C.c_int, [c_p, C.c_int, c_p, c_i64, C.c_int, C.c_float, c_p, c_p, c_p, c_p]),
    "unetb200_ce_dice_bwd": (C.c_int, [c_p, C.c_int, c_p, c_i64, C.c_int, c_p, c_p, c_p, c_p]),
    "unetb200_bce_dice_work_bytes": (c_i64, [c_i64]),
    "unetb200_bce_dice_fwd": (C.c_int, [c_p, C.c_int, c_p, C.c_int, c_i64, C.c_float, c_p, c_p, c_p, c_p]),
    "unetb200_bce_dice_bwd": (C.c_int, [c_p, C.c_int, c_p, C.c_int, c_i64, c_p, c_p, c_p, c_p]),
    "unetb200_dice_fwd": (C.c_int, [c_p, c_p, c_i64, c_i64, C.c_float, c_p, c_p, c_p, c_p]),
    "unetb200_dice_bwd": (C.c_int, [c_p, c_p, c_i64, c_i64, C.c_float, c_p, c_p, c_p, c_p]),
    "unetb200_boundary_loss": (C.c_int, [c_p, C.c_int, c_i64, c_i64, c_i64, c_p, C.c_int, c_i64, c_i64, c_i64,
                                         C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_float, c_p, c_p, c_p]),
    "unetb200_boundary_work_bytes": (c_i64, []),
    "unetb200_grad_sqnorm": (C.c_int, [c_p, c_p, C.c_int, c_p, c_p]),
    "unetb200_rmsprop_step": (C.c_int, [c_p, c_p, c_p, c_p, c_p, C.c_int, c_p, C.c_float, C.c_float, C.c_float, C.c_float,
                                        C.c_float, C.c_float, C.c_int, c_p]),
    "unetb200_grad_sqnorm_amp": (C.c_int, [c_p, c_p, C.c_int, c_p, c_p, c_p, c_p]),
    "unetb200_rmsprop_step_amp": (C.c_int, [c_p, c_p, c_p, c_p, c_p, c_p, C.c_int, c_p, C.c_float, c_p, c_p, c_p,
                                            C.c_float, C.c_float, C.c_float, C.c_float, C.c_int, c_p]),
    "unetb200_eval_counts": (C.c_int, [c_p, C.c_int, c_i64, c_i64, c_i64, c_i64, c_p, C.c_int, C.c_int, C.c_int,
                                       C.c_int, C.c_int, C.c_int, C.c_int, c_p, C.c_int, c_p, C.c_float, c_p, c_p]),
    "unetb200_resize_argmax": (C.c_int, [c_p, C.c_int, c_i64, c_i64, c_i64, c_i64] + [C.c_int] * 6 + [c_p, C.c_int, c_p]),
    "unetb200_preprocess_image_u8": (C.c_int, [c_p, C.c_int, C.c_int, C.c_int, C.c_int, c_p, C.c_int, c_p, c_p, c_p]),
    "unetb200_preprocess_mask_u8": (C.c_int, [c_p, C.c_int, C.c_int, C.c_int, c_p, C.c_int, c_p, c_p, c_p]),
}

_lib = None


class UnetB200Error(RuntimeError):
    pass


def load():
    """Load the shared library (once).  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise UnetB200Error(
            f"{LIB_PATH} not found: build it with `make -C "
            f"{os.path.join(os.path.dirname(_HERE), 'csrc')}` (or __graft_entry__.build()). "
            "There is no PyTorch/CPU fallback for the UNet hot path.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)          # AttributeError if the .so lacks a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int, what: str = ""):
    if rc == 0:
        return
    msg = load().unetb200_last_error().decode("utf-8", "replace")
    text = f"libunetb200 {what}: {msg} (status {rc})"
    if rc == E_INVALID:
        raise ValueError(text)
    if rc == E_NOMEM:
        import torch
        raise torch.cuda.OutOfMemoryError(text)
    raise UnetB200Error(text)
