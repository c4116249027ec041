"""CPU: every C-ABI entry point that turns a dtype code into a kernel's template arguments rejects an unknown code
before it touches the device: UNETB200_E_INVALID and the same unetb200_last_error() text, whatever else the call
gets right.  An unknown code must never fall through to the fp32 (or int64) kernels."""
import ctypes

import pytest

from unetb200 import _lib

BAD = 7                    # no dtype has this code
F32, BF16, I64 = _lib.F32, _lib.BF16, _lib.I64
P = 4096                   # a non-null, 16-byte-aligned pointer; validation fails before anything reads it
S = None                   # default stream
B, H, W, C = 2, 8, 8, 16
NPIX = B * H * W


def _gconv(dtype):
    d = _lib.GConv(dtype=dtype, algo=_lib.ALGO_AUTO, B=B, Hm=H, Wm=W, Cin=C, ntaps=9, in_scale=1, Hin=H, Win=W,
                   ld_in=C, N=C, nquad=1, out_scale=1, Hout=H, Wout=W, ld_out=C)
    for t in range(9):
        d.tap_dy[t], d.tap_dx[t] = t // 3 - 1, t % 3 - 1
    return ctypes.byref(d)


def _pack_job():
    return ctypes.byref(_lib.PackJob(src=P, dst=P, n0=C, n1=9, n2=C, s0=1, s1=C, s2=9 * C, off=0))


# (entry point, arguments with BAD in the position under test, unetb200_last_error() text)
CASES = [
    ("bn_relu_apply", lambda: (P, C, P, P, P, C, None, 0, BAD, B, H, W, C, S), "unsupported dtype 7"),
    ("maxpool2_fwd", lambda: (P, C, P, C, BAD, B, H, W, C, S), "unsupported dtype 7"),
    ("maxpool2_bwd", lambda: (P, C, P, C, P, C, 0, BAD, B, H, W, C, S), "unsupported dtype 7"),
    ("maxpool2_bwd_bnreduce", lambda: (P, C, P, C, P, C, P, C, P, P, P, P, P, BAD, B, H, W, C, S),
     "unsupported dtype 7"),
    ("bn_relu_bwd_reduce", lambda: (P, C, P, C, P, P, P, P, P, BAD, B, H, W, C, S), "unsupported dtype 7"),
    ("bn_relu_bwd_apply", lambda: (P, C, P, C, P, P, P, P, P, P, C, BAD, B, H, W, C, S), "unsupported dtype 7"),
    ("upsample2x_fwd", lambda: (P, C, P, C, BAD, B, H, W, C, 2 * H, 2 * W, 0, 0, S), "unsupported dtype 7"),
    ("upsample2x_bwd", lambda: (P, C, P, C, BAD, B, H, W, C, 2 * H, 2 * W, 0, 0, S), "unsupported dtype 7"),
    ("gather_nhwc", lambda: (P, BAD, H * W * C, 1, W * C, C, P, BF16, C, B, C, H, W, S), "unsupported dtype 7"),
    ("gather_nhwc", lambda: (P, F32, H * W * C, 1, W * C, C, P, BAD, C, B, C, H, W, S), "unsupported dtype 7"),
    ("copy_channels", lambda: (P, BAD, C, P, BF16, C, NPIX, C, S), "unsupported dtype 7"),
    ("copy_channels", lambda: (P, F32, C, P, BAD, C, NPIX, C, S), "unsupported dtype 7"),
    ("zero_channels", lambda: (P, BAD, C, NPIX, C, S), "unsupported dtype 7"),
    ("add_channels", lambda: (P, C, P, C, BAD, NPIX, C, S), "unsupported dtype 7"),
    ("channel_sum", lambda: (P, BAD, C, NPIX, C, P, P, S), "unsupported dtype 7"),
    ("ce_dice_fwd", lambda: (P, BAD, P, NPIX, 2, 1e-6, P, P, P, S), "ce_dice_fwd: dtype"),
    ("ce_dice_bwd", lambda: (P, BAD, P, NPIX, 2, P, P, P, S), "ce_dice_bwd: dtype"),
    ("bce_dice_fwd", lambda: (P, BAD, P, F32, NPIX, 1e-6, P, P, P, S), "bce_dice_fwd: dtype"),
    ("bce_dice_fwd", lambda: (P, BF16, P, BAD, NPIX, 1e-6, P, P, P, S), "bce_dice_fwd: target dtype"),
    ("bce_dice_bwd", lambda: (P, BAD, P, F32, NPIX, P, P, P, S), "bce_dice_bwd: dtype"),
    ("bce_dice_bwd", lambda: (P, BF16, P, BAD, NPIX, P, P, P, S), "bce_dice_bwd: target dtype"),
    ("boundary_loss", lambda: (P, BAD, H * W, W, 1, P, F32, H * W, W, 1, B, H, W, 2, 1.0, 1.0, P, P, S),
     "boundary_loss: pred dtype"),
    ("boundary_loss", lambda: (P, F32, H * W, W, 1, P, BAD, H * W, W, 1, B, H, W, 2, 1.0, 1.0, P, P, S),
     "boundary_loss: target dtype"),
    ("eval_counts", lambda: (P, BAD, H * W * 2, 1, W * 2, 2, P, I64, B, 2, H, W, 1, 0, P, I64, P, 1e-6, None, S),
     "eval_counts: logits dtype"),
    ("eval_counts", lambda: (P, BF16, H * W * 2, 1, W * 2, 2, P, BAD, B, 2, H, W, 1, 0, P, I64, P, 1e-6, None, S),
     "eval_counts: target dtype"),
    ("eval_counts", lambda: (P, BF16, H * W * 2, 1, W * 2, 2, P, I64, B, 2, H, W, 1, 0, P, BAD, P, 1e-6, None, S),
     "eval_counts: prediction dtype must be int64 or uint8"),
    ("resize_argmax", lambda: (P, BAD, H * W * 2, 1, W * 2, 2, B, 2, H, W, 2 * H, 2 * W, P, I64, S),
     "resize_argmax: logits dtype"),
    ("resize_argmax", lambda: (P, BF16, H * W * 2, 1, W * 2, 2, B, 2, H, W, 2 * H, 2 * W, P, BAD, S),
     "resize_argmax: output dtype"),
    ("outconv_fwd", lambda: (P, C, P, P, P, BAD, NPIX, C, 2, S), "outconv_fwd: dtype"),
    ("outconv_bwd", lambda: (P, C, P, P, P, C, P, P, P, BAD, NPIX, C, 2, S), "outconv_bwd: dtype"),
    ("outconv_bwd_bnbwd", lambda: (P, C, P, P, P, C, P, P, P, P, C, P, P, BAD, NPIX, C, 2, S),
     "outconv_bwd_bnbwd: shape not covered (query _supported first and run outconv_bwd + bn_relu_bwd_reduce)"),
    ("sa_forward", lambda: (P, C, P, P, P, P, C, BAD, B, H, W, C, S), "sa_forward: dtype"),
    ("sa_backward", lambda: (P, C, P, C, P, P, P, P, C, P, P, BAD, B, H, W, C, S), "sa_backward: dtype"),
    ("pack_weights", lambda: (P, P, BAD, C, 9, C, 1, C, 9 * C, 0, S), "pack_weights: dtype"),
    ("pack_weights_multi", lambda: (_pack_job(), 1, BAD, S), "pack_weights_multi: dtype"),
    ("gconv_fprop", lambda: (_gconv(BAD), P, P, None, P, None, None, None, S), "gconv: dtype 7"),
]


@pytest.mark.parametrize("name,args,message", CASES, ids=[f"{n}-{i}" for i, (n, _, _) in enumerate(CASES)])
def test_unknown_dtype_code_is_rejected(name, args, message):
    lib = _lib.load()
    rc = getattr(lib, "unetb200_" + name)(*args())
    assert rc == _lib.E_INVALID
    assert lib.unetb200_last_error().decode() == message

