"""Tensor-level wrappers over the C ABI: they only marshal ``data_ptr()``, shapes, strides and the
current CUDA stream.  PyTorch is used for device memory (``torch.empty`` through the caching
allocator, so OOM surfaces as ``torch.cuda.OutOfMemoryError``) and streams -- never for arithmetic.

Activation convention: a logical [B, C, H, W] tensor whose strides are (H*W*ld, 1, W*ld, ld) is
"NHWC with pixel stride ld"; ld > C is a channel slice of a wider NHWC buffer.

Every wrapper goes through :func:`_run`, which counts kernel launches (``LAUNCHES``, bench.py's
``gpu_launches``) and, inside ``with profile() as rec:``, brackets the call with CUDA events on the
launching stream and records its algorithmic FLOPs / bytes (bench.py's ``roofline``).
"""
from __future__ import annotations

import contextlib
import ctypes as C
import os

import torch

from . import _lib, backward_pass
from ._lib import ALGO_AUTO, ALGO_SIMT, ALGO_TC, BF16, F32, I64, GConv  # noqa: F401

_DT = {torch.float32: F32, torch.bfloat16: BF16}
_ESZ = {torch.float32: 4, torch.bfloat16: 2}

LAUNCHES = 0
_PROFILE = None


@contextlib.contextmanager
def profile():
    """Collect (name, start_event, end_event, flops, bytes) per C-ABI call."""
    global _PROFILE
    prev, _PROFILE = _PROFILE, []
    try:
        yield _PROFILE
    finally:
        _PROFILE = prev


def summarize_profile(rec):
    """{name: dict(ms, calls, flops, bytes)} -- call after torch.cuda.synchronize()."""
    out = {}
    for name, s, e, flops, nbytes in rec:
        d = out.setdefault(name, dict(ms=0.0, calls=0, flops=0.0, bytes=0.0))
        d["ms"] += s.elapsed_time(e)
        d["calls"] += 1
        d["flops"] += flops
        d["bytes"] += nbytes
    return out


def lib():
    return _lib.load()


# torch.cuda.current_stream() costs ~18 us of Python per call (device-index plumbing, an environment lookup in
# is_available); the light variants issue ~230 launches per step and are launch-bound when run eagerly
_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)
_cur_device = getattr(torch._C, "_cuda_getDevice", None)


def _stream():
    if _raw_stream is not None and _cur_device is not None:
        return C.c_void_p(_raw_stream(_cur_device()))
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _run(name, fn, *args, kernels=1, flops=0.0, nbytes=0.0):
    global LAUNCHES
    if _PROFILE is not None:
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        rc = fn(*args)
        e.record()
        _PROFILE.append([name, s, e, flops, nbytes])
    else:
        rc = fn(*args)
    LAUNCHES += kernels
    _lib.check(rc, name)


def _p(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def _prow(t, i):
    """pointer to row i of a 2-D tensor (no view tensor is created: ~3 us each on the launch path)"""
    return C.c_void_p(t.data_ptr() + i * t.stride(0) * t.element_size())


def dt(t):
    try:
        return _DT[t.dtype]
    except KeyError:
        raise ValueError(f"unetb200: unsupported dtype {t.dtype}") from None


def require_cuda(t, what):
    if not t.is_cuda:
        raise RuntimeError(
            f"unetb200.{what}: the B200 hot path runs on CUDA tensors only (got a {t.device} tensor); "
            "there is deliberately no CPU fallback -- move the model and inputs to the GPU.")


# ------------------------------------------------------------------------------------------------
# NHWC views
# ------------------------------------------------------------------------------------------------
def nhwc_ld(t):
    """Pixel stride of a logical [B,C,H,W] tensor if it is NHWC-with-ld, else None."""
    if t.dim() != 4:
        return None
    B, Cc, H, W = t.shape
    sb, sc, sh, sw = t.stride()
    if Cc > 1 and sc != 1:
        return None
    if W > 1:
        ld = sw
    elif H > 1:
        ld = sh
    elif B > 1:
        ld = sb
    else:
        ld = Cc
    if ld < Cc:
        return None
    if H > 1 and sh != W * ld:
        return None
    if B > 1 and sb != H * W * ld:
        return None
    return ld


def empty_nhwc(B, Cc, H, W, dtype, device):
    """Logical [B,C,H,W], physically NHWC contiguous."""
    return torch.empty((B, H, W, Cc), dtype=dtype, device=device).permute(0, 3, 1, 2)


def channel_slice(buf, c0, Cc):
    """Alias of channels [c0, c0+Cc) of an NHWC buffer, without an autograd view relation."""
    B, Ct, H, W = buf.shape
    ld = nhwc_ld(buf)
    out = buf.new_empty(0)
    out.set_(buf.untyped_storage(), buf.storage_offset() + c0, (B, Cc, H, W), (H * W * ld, 1, W * ld, ld))
    return out


def to_nhwc(x, dtype, packed=False):
    """Any-strided logical NCHW tensor -> NHWC of `dtype` (no copy if it already is; with
    packed=True the pixel stride must equal C)."""
    ld = nhwc_ld(x)
    if x.dtype == dtype and ld is not None and (not packed or ld == x.shape[1]):
        return x
    if x.dtype not in _DT:
        x = x.float()
    B, Cc, H, W = x.shape
    out = empty_nhwc(B, Cc, H, W, dtype, x.device)
    sn, sc, sh, sw = x.stride()
    _run("gather_nhwc", lib().unetb200_gather_nhwc, _p(x), dt(x), sn, sc, sh, sw, _p(out), _DT[dtype], Cc, B, Cc, H,
         W, _stream(), nbytes=x.numel() * (x.element_size() + _ESZ[dtype]))
    return out


def copy_channels(src, dst):
    B, Cc, H, W = src.shape
    _run("copy_channels", lib().unetb200_copy_channels, _p(src), dt(src), nhwc_ld(src), _p(dst), dt(dst),
         nhwc_ld(dst), B * H * W, Cc, _stream(), nbytes=src.numel() * (src.element_size() + dst.element_size()))


def zero_channels(dst):
    B, Cc, H, W = dst.shape
    _run("zero_channels", lib().unetb200_zero_channels, _p(dst), dt(dst), nhwc_ld(dst), B * H * W, Cc, _stream(),
         nbytes=dst.numel() * dst.element_size())


def add_channels_(a, b):
    B, Cc, H, W = a.shape
    _run("add_channels", lib().unetb200_add_channels, _p(a), nhwc_ld(a), _p(b), nhwc_ld(b), dt(a), B * H * W, Cc,
         _stream(), nbytes=3 * a.numel() * a.element_size())
    return a


def channel_sum(g, out=None):
    B, Cc, H, W = g.shape
    acc = torch.empty(Cc, dtype=torch.float64, device=g.device)
    if out is None:
        out = torch.empty(Cc, dtype=torch.float32, device=g.device)
    _run("channel_sum", lib().unetb200_channel_sum, _p(g), dt(g), nhwc_ld(g), B * H * W, Cc, _p(acc), _p(out),
         _stream(), kernels=2, nbytes=g.numel() * g.element_size())
    return out


def f64_to_f32(src, out=None):
    """fp64 vector (a slice of conv-epilogue column sums) -> fp32 parameter gradient"""
    if out is None:
        out = torch.empty(src.numel(), dtype=torch.float32, device=src.device)
    _run("bias_from_colsum", lib().unetb200_f64_to_f32, _p(src), _p(out), src.numel(), _stream())
    return out


# ------------------------------------------------------------------------------------------------
# generalised convolution
# ------------------------------------------------------------------------------------------------
TAPS3 = [(kh - 1, kw - 1) for kh in range(3) for kw in range(3)]
TAPS1 = [(0, 0)]
TAPS_Q = [(0, 0), (0, 1), (1, 0), (1, 1)]
_ALGO_NAME = {ALGO_SIMT: "simt", ALGO_TC: "tc"}


_FORCED_ALGO = {"simt": ALGO_SIMT, "tc": ALGO_TC}.get(os.environ.get("UNETB200_ALGO", "").lower(), None)


def forced_algo():
    """UNETB200_ALGO=simt|tc (read once at import): every convolution on one engine, for A/B runs."""
    return _FORCED_ALGO


def make_gconv(dtype, algo, B, Hm, Wm, Cin, taps, in_scale, in_off, Hin, Win, ld_in, N, nquad, out_scale, out_off,
               Hout, Wout, ld_out):
    d = GConv()
    d.dtype = dtype
    fa = forced_algo()
    d.algo = fa if fa is not None else algo
    if dtype == F32 and d.algo == _lib.ALGO_PREFER_TC and Cin < 16 and x3_mode():
        # fp32 exactness mode: layers too narrow for the 3-term split (x3_active needs C_in >= 16) stay on the exact
        # CUDA-core kernels instead of the plain-TF32 narrow kernel
        d.algo = ALGO_SIMT
    d.B, d.Hm, d.Wm, d.Cin, d.ntaps = B, Hm, Wm, Cin, len(taps)
    for i, (dy, dx) in enumerate(taps):
        d.tap_dy[i], d.tap_dx[i] = dy, dx
    d.in_scale, d.in_off_y, d.in_off_x = in_scale, in_off[0], in_off[1]
    d.Hin, d.Win, d.ld_in = Hin, Win, ld_in
    d.N, d.nquad, d.out_scale = N, nquad, out_scale
    d.out_off_y, d.out_off_x = out_off
    d.Hout, d.Wout, d.ld_out = Hout, Wout, ld_out
    return d


def _shape_tag(d):
    """Per-layer profile names when UNETB200_PROFILE_SHAPES is set (bench.py --per-layer)."""
    if _PROFILE is None or not os.environ.get("UNETB200_PROFILE_SHAPES"):
        return ""
    return f"[M={d.B * d.Hm * d.Wm},N={d.N},K={d.ntaps * d.Cin}]"


def gconv_flops(d):
    """Algorithmic FLOPs of one launch: 2*M*N*K (SURVEY.md section 8d)."""
    return 2.0 * d.B * d.Hm * d.Wm * d.N * d.ntaps * d.Cin


def gconv_bytes(d, es):
    """Algorithmic bytes of one launch: every input element, weight and output element once (the taps of a 3x3
    window are served from L2 / shared memory, not HBM)."""
    m_in = d.B * d.Hin * d.Win if d.in_scale == 1 else d.B * d.Hm * d.Wm * d.ntaps
    return float(es) * (m_in * d.Cin + d.B * d.Hm * d.Wm * d.N + d.N * d.ntaps * d.Cin)


# ---- fp32 exactness mode on the tensor cores: 3xTF32 ---------------------------------------------------------
def x3_mode():
    return os.environ.get("UNET_B200_PRECISION", "").lower() == "tf32x3"


def x3_active(d):
    """UNET_B200_PRECISION=tf32x3: fp32 convolutions with C_in >= 16 run as ONE tcgen05 kind::tf32 implicit GEMM over
    3*C_in channels [hi | lo | hi] x [hi | hi | lo] (unetb200_split_tf32), i.e. hi*hi + lo*hi + hi*lo with fp32
    accumulation -- fp32-level results (~1e-6) at a third of the TF32 rate.  The first layer (C_in <= 4) and OutConv
    are exact fp32 CUDA-core kernels in every mode."""
    return d.dtype == F32 and d.algo in (ALGO_TC, _lib.ALGO_PREFER_TC) and d.Cin >= 16 and x3_mode()


def x3_split(x):
    """NHWC fp32 [B,C,H,W] (any pixel stride) -> packed NHWC [B,3C,H,W] = [hi | lo | hi]."""
    B, Cc, H, W = x.shape
    out = empty_nhwc(B, 3 * Cc, H, W, torch.float32, x.device)
    _run("split_tf32", lib().unetb200_split_tf32, _p(x), nhwc_ld(x), _p(out), B * H * W, Cc, 0, _stream(),
         nbytes=16.0 * x.numel())
    return out


def x3_split_rows(wp, rows, Cc):
    """packed weights [rows][C] (rows = (n, tap)) -> [rows][3C] = [hi | hi | lo]."""
    out = torch.empty((rows * 3 * Cc,), dtype=torch.float32, device=wp.device)
    _run("split_tf32_w", lib().unetb200_split_tf32, _p(wp), Cc, _p(out), rows, Cc, 1, _stream(), nbytes=16.0 * rows * Cc)
    return out


def _x3_desc(d, ld_in=None, ld_out=None, triple=True):
    d3 = GConv.from_buffer_copy(d)
    if triple:
        d3.Cin = 3 * d.Cin
    if ld_in is not None:
        d3.ld_in = ld_in
    if ld_out is not None:
        d3.ld_out = ld_out
    return d3


def gconv_fprop(d, x, wp, bias, y, stats, kind="fprop", x_split=None):
    used = C.c_int(0)
    ws = None
    flops, nbytes = gconv_flops(d), gconv_bytes(d, 2 if d.dtype == BF16 else 4)
    tag = _shape_tag(d)
    if x3_active(d):
        xs = x_split if x_split is not None else x3_split(x)
        wp = x3_split_rows(wp, d.N * d.ntaps, d.Cin)
        d = _x3_desc(d, ld_in=3 * d.Cin)
        x = xs
        kind = kind + "_x3"
    if stats is not None:
        n = lib().unetb200_gconv_stats_workspace(C.byref(d))
        if n < 0:
            _lib.check(-1, "gconv_stats_workspace")
        ws = torch.empty(n, dtype=torch.float32, device=x.device)
    _run(f"conv_{kind}", lib().unetb200_gconv_fprop, C.byref(d), _p(x), _p(wp), _p(bias), _p(y), _p(stats), _p(ws),
         C.byref(used), _stream(), kernels=2 if stats is not None else 1, flops=flops, nbytes=nbytes)
    if _PROFILE is not None:
        _PROFILE[-1][0] = f"conv_{kind}_{_ALGO_NAME.get(used.value, '?')}" + tag
    return used.value


def gconv_fprop_affine_relu_supported(d, x, wp, z):
    if x3_active(d):
        d = _x3_desc(d, ld_in=3 * d.Cin)
    return bool(lib().unetb200_gconv_fprop_affine_relu_supported(C.byref(d), _p(x), _p(wp), _p(z)))


def gconv_fprop_affine_relu_pool_supported(d, x, wp, z, pooled):
    return (not x3_active(d)) and bool(lib().unetb200_gconv_fprop_affine_relu_pool_supported(
        C.byref(d), _p(x), _p(wp), _p(z), _p(pooled), nhwc_ld(pooled)))


def gconv_fprop_affine_relu(d, x, wp, coefs, z, pooled=None):
    """z = relu(conv(x, wp) * scale + shift) in the tcgen05 epilogue (inference; coefs rows 2, 3 = scale, shift);
    pooled (query gconv_fprop_affine_relu_pool_supported first) = MaxPool2d(2)(z) from the same epilogue."""
    flops, nbytes = gconv_flops(d), gconv_bytes(d, 2 if d.dtype == BF16 else 4)
    tag = _shape_tag(d)
    if pooled is not None:
        _run("conv_fprop_bnfold", lib().unetb200_gconv_fprop_affine_relu_pool, C.byref(d), _p(x), _p(wp), _prow(coefs, 2),
             _p(z), _p(pooled), nhwc_ld(pooled), _stream(), flops=flops,
             nbytes=nbytes + float(pooled.numel()) * pooled.element_size())
        if _PROFILE is not None:
            _PROFILE[-1][0] = "conv_fprop_bnfold_tc" + tag
        return
    if x3_active(d):
        x = x3_split(x)
        wp = x3_split_rows(wp, d.N * d.ntaps, d.Cin)
        d = _x3_desc(d, ld_in=3 * d.Cin)
    _run("conv_fprop_bnfold", lib().unetb200_gconv_fprop_affine_relu, C.byref(d), _p(x), _p(wp), _prow(coefs, 2), _p(z),
         _stream(), flops=flops, nbytes=nbytes)
    if _PROFILE is not None:
        _PROFILE[-1][0] = "conv_fprop_bnfold_tc" + tag


def gconv_fprop_affine_relu_outconv_supported(d, x, wp, ncls):
    return (not x3_active(d)) and bool(lib().unetb200_gconv_fprop_affine_relu_outconv_supported(C.byref(d), _p(x), _p(wp), ncls))


def gconv_fprop_affine_relu_outconv(d, x, wp, coefs, oc_w, oc_b, logits):
    """logits = OutConv(relu(conv(x, wp) * scale + shift)) in ONE kernel (inference; the activation is never written)."""
    flops, tag = gconv_flops(d), _shape_tag(d)
    ncls = oc_w.shape[0]
    es = 2 if d.dtype == BF16 else 4
    _run("conv_fprop_bnfold", lib().unetb200_gconv_fprop_affine_relu_outconv, C.byref(d), _p(x), _p(wp), _prow(coefs, 2),
         _p(oc_w), _p(oc_b), _p(logits), ncls, _stream(), flops=flops,
         nbytes=float(es) * d.B * d.Hin * d.Win * d.Cin + float(es) * d.B * d.Hm * d.Wm * ncls)
    if _PROFILE is not None:
        _PROFILE[-1][0] = "conv_fprop_bnfold_tc" + tag


def gconv_dgrad_bnbwd_supported(d, g, wp, gx):
    return (not x3_active(d)) and bool(lib().unetb200_gconv_dgrad_bnbwd_supported(C.byref(d), _p(g), _p(wp), _p(gx)))


def gconv_dgrad_bnbwd(d, g, wp, gx, yprev, coefs_prev):
    """gx = dgrad conv; returns fp64 sums[2, C] of the BatchNorm + ReLU backward of the layer whose raw output is
    `yprev` (gx is the gradient of relu(bn(yprev))): the reduce pass rides in the tcgen05 epilogue."""
    flops, nbytes = gconv_flops(d), gconv_bytes(d, 2 if d.dtype == BF16 else 4)
    tag = _shape_tag(d)
    sums = torch.zeros((2, d.N), dtype=torch.float64, device=g.device)
    n = lib().unetb200_gconv_stats_workspace(C.byref(d))
    if n < 0:
        _lib.check(-1, "gconv_stats_workspace")
    ws = torch.empty(n, dtype=torch.float32, device=g.device)
    if not coefs_prev.is_contiguous():
        raise ValueError("unetb200: BatchNorm coefficients must be a contiguous [4, C] tensor")
    _run("conv_dgrad_tc" + tag, lib().unetb200_gconv_dgrad_bnbwd, C.byref(d), _p(g), _p(wp), _p(gx), _p(yprev),
         nhwc_ld(yprev), _p(coefs_prev), _p(sums), _p(ws), _stream(), kernels=2, flops=flops,
         nbytes=nbytes + float(yprev.numel()) * yprev.element_size())
    return sums


# Switches of the backward pass's bookkeeping (unetb200.backward_pass reads them at each use, so a script or test may
# flip them here): batched split reductions; the side stream at all; weight gradients on it -- OFF by default: it paid
# (+4 %) while the wgrad grids had a nearly empty third wave for the BatchNorm kernels to fill; with wave-exact split
# counts the serial order is 1-2 % faster.
DEFER_REDUCE = os.environ.get("UNETB200_DEFER_REDUCE", "1") != "0"
_SIDE_ON = os.environ.get("UNETB200_SIDE_STREAM", "1") != "0"
_WGRAD_SIDE = os.environ.get("UNETB200_WGRAD_STREAM", "0") != "0"


def _wgrad_once(d, x, gy, dst, st, sc, sn, sq, accumulate, flops, tag, defer=False):
    splits, used = C.c_int(0), C.c_int(0)
    _lib.check(lib().unetb200_gconv_wgrad_plan(C.byref(d), C.byref(splits), C.byref(used)), "gconv_wgrad_plan")
    K = d.ntaps * d.Cin
    partials = torch.empty(splits.value * K * d.N, dtype=torch.float32, device=x.device)
    d2 = GConv.from_buffer_copy(d)
    d2.algo = used.value
    es = 2 if d.dtype == BF16 else 4
    _run(f"conv_wgrad_{_ALGO_NAME.get(used.value, '?')}" + tag, lib().unetb200_gconv_wgrad, C.byref(d2), _p(x), _p(gy),
         _p(partials), splits.value, _stream(), flops=flops,
         nbytes=float(es) * d.B * (d.Hin * d.Win * d.Cin + d.Hout * d.Wout * (d.N // d.nquad)) + 4.0 * K * d.N)
    if defer and not accumulate and backward_pass.defer_reduce(
            (partials, dst.data_ptr(), st, sc, sq, sn, splits.value, d.ntaps, d.Cin, d.N, d.N // d.nquad), defer):
        return used.value
    _run("wgrad_reduce", lib().unetb200_wgrad_reduce, _p(partials), splits.value, d.ntaps, d.Cin, d.N,
         d.N // d.nquad, _p(dst), st, sc, sq, sn, 1 if accumulate else 0, _stream(),
         nbytes=4.0 * K * d.N * (splits.value + 1))
    return used.value


def gconv_wgrad(d, x, gy, dst, st, sc, sn, sq=0, x_split=None, gy_split=None, defer=False):
    """dst (parameter layout, fp32) = weight gradient; dst[t*st + c*sc + q*sq + co*sn], n = q*Cq + co.
    defer="call": the split reduction joins the one launch made when the enclosing backward_pass.reductions_at_return
    block ends (made at once outside such a block); defer="pass": nothing but the data-parallel reducer reads dst
    before the end of the backward pass -- the reduction joins the one launch at the end of the pass
    (backward_pass.defer_reduce)."""
    if not x3_active(d):
        return _wgrad_once(d, x, gy, dst, st, sc, sn, sq, False, gconv_flops(d), _shape_tag(d), defer=defer)
    # 3xTF32: dW = hi(x)^T hi(g) + lo(x)^T hi(g) + hi(x)^T lo(g), the last two accumulated by the split reduction
    xs = x_split if x_split is not None else x3_split(x)
    gs = gy_split if gy_split is not None else x3_split(gy)
    Cg = gy.shape[1]
    d2 = _x3_desc(d, ld_in=3 * d.Cin, ld_out=3 * Cg, triple=False)
    x_hi, x_lo = channel_slice(xs, 0, d.Cin), channel_slice(xs, d.Cin, d.Cin)
    g_hi, g_lo = channel_slice(gs, 0, Cg), channel_slice(gs, Cg, Cg)
    tag = "_x3" + _shape_tag(d)
    used = _wgrad_once(d2, x_hi, g_hi, dst, st, sc, sn, sq, False, gconv_flops(d), tag)
    _wgrad_once(d2, x_lo, g_hi, dst, st, sc, sn, sq, True, 0.0, tag)
    _wgrad_once(d2, x_hi, g_lo, dst, st, sc, sn, sq, True, 0.0, tag)
    return used


# ------------------------------------------------------------------------------------------------
# BatchNorm / ReLU / pooling
# ------------------------------------------------------------------------------------------------
def bn_finalize(stats, count, gamma, beta, eps, momentum, running_mean, running_var, Cc, num_batches_tracked=None):
    """`num_batches_tracked`: the module's int64 step counter, incremented by the same launch when given."""
    dev = stats.device
    coefs = torch.empty((4, Cc), dtype=torch.float32, device=dev)   # mean, invstd, scale, shift
    nbt = num_batches_tracked
    if nbt is not None and not (nbt.dtype == torch.int64 and nbt.is_cuda and nbt.numel() == 1):
        nbt.add_(1)                                                  # a counter the kernel cannot reach (never on the path)
        nbt = None
    _run("bn_finalize", lib().unetb200_bn_finalize_track, _p(stats), count, _p(gamma), _p(beta), eps, momentum,
         _p(running_mean), _p(running_var), _prow(coefs, 0), _prow(coefs, 1), _prow(coefs, 2), _prow(coefs, 3), _p(nbt), Cc, _stream())
    if nbt is not None:
        torch._C._increment_version([nbt])
    return coefs


def bn_sync_finalize(peer, stats, count, gamma, beta, eps, momentum, running_mean, running_var, Cc,
                     num_batches_tracked=None):
    """bn_finalize on the statistics of every rank of `peer` (a ddp.BNPeerGroup): one single-CTA exchange launch."""
    peer.check()
    coefs = torch.empty((4, Cc), dtype=torch.float32, device=stats.device)
    nbt = num_batches_tracked
    if nbt is not None and not (nbt.dtype == torch.int64 and nbt.is_cuda and nbt.numel() == 1):
        nbt.add_(1)
        nbt = None
    _run("bn_sync_finalize", lib().unetb200_bn_sync_finalize, peer.handle, _p(stats), count, _p(gamma), _p(beta), eps,
         momentum, _p(running_mean), _p(running_var), _prow(coefs, 0), _prow(coefs, 1), _prow(coefs, 2),
         _prow(coefs, 3), _p(nbt), Cc, _stream())
    if nbt is not None:
        torch._C._increment_version([nbt])
    return coefs


def bn_sync_bwd_finalize(peer, sums, count, dgamma, dbeta, coef):
    """bn_bwd_finalize (training) with the coefficients from the sums of every rank of `peer`; dgamma / dbeta local."""
    peer.check()
    _run("bn_sync_bwd_finalize", lib().unetb200_bn_sync_bwd_finalize, peer.handle, _p(sums), count, _p(dgamma),
         _p(dbeta), _p(coef), coef.shape[1], _stream())


def bn_eval_coeffs(gamma, beta, running_mean, running_var, eps, Cc):
    coefs = torch.empty((4, Cc), dtype=torch.float32, device=running_mean.device)
    _run("bn_eval_coeffs", lib().unetb200_bn_eval_coeffs, _p(gamma), _p(beta), _p(running_mean), _p(running_var),
         eps, _prow(coefs, 2), _prow(coefs, 3), _prow(coefs, 0), _prow(coefs, 1), Cc, _stream())
    return coefs


def bn_relu_apply(y, coefs, z, pooled=None):
    B, Cc, H, W = y.shape
    es = y.element_size()
    _run("bn_relu_apply_pool" if pooled is not None else "bn_relu_apply", lib().unetb200_bn_relu_apply, _p(y),
         nhwc_ld(y), _prow(coefs, 2), _prow(coefs, 3), _p(z), nhwc_ld(z), _p(pooled),
         nhwc_ld(pooled) if pooled is not None else 0, dt(y), B, H, W, Cc, _stream(),
         nbytes=y.numel() * es * (2.25 if pooled is not None else 2.0))


def maxpool2_fwd(x, p):
    B, Cc, H, W = x.shape
    _run("maxpool2_fwd", lib().unetb200_maxpool2_fwd, _p(x), nhwc_ld(x), _p(p), nhwc_ld(p), dt(x), B, H, W, Cc,
         _stream(), nbytes=x.numel() * x.element_size() * 1.25)


def maxpool2_bwd(x, gp, gx, accumulate):
    B, Cc, H, W = x.shape
    _run("maxpool2_bwd", lib().unetb200_maxpool2_bwd, _p(x), nhwc_ld(x), _p(gp), nhwc_ld(gp), _p(gx), nhwc_ld(gx),
         1 if accumulate else 0, dt(x), B, H, W, Cc, _stream(),
         nbytes=x.numel() * x.element_size() * (3.25 if accumulate else 2.25))


# Measured at C2 (4 encoder stages, B = 16): fused 1.18 ms against 0.54 ms + 0.38 ms for the separate reduction
# passes -- ~110 registers per thread (four coefficient vectors + two sum vectors on top of the pool's own state)
# leave two blocks per SM and the stream runs at 0.55 of the copy peak -- so the fused form is opt-in; it stays tested.
POOL_BNBWD_FUSE = os.environ.get("UNETB200_POOL_BNBWD_FUSE", "0") != "0" and os.environ.get("UNETB200_NO_BNBWD_FUSE") is None


def maxpool2_bwd_bnreduce(x, gp, gx, y, coefs):
    """gx += max-pool scatter of gp (in place), and the fp64 sums[2, C] of the BatchNorm + ReLU backward of the layer
    whose raw output is y (x = relu(bn(y)), gx its now complete output gradient) from the same pass."""
    B, Cc, H, W = x.shape
    sums = torch.zeros((2, Cc), dtype=torch.float64, device=x.device)
    _run("maxpool2_bwd", lib().unetb200_maxpool2_bwd_bnreduce, _p(x), nhwc_ld(x), _p(gp), nhwc_ld(gp), _p(gx), nhwc_ld(gx),
         _p(y), nhwc_ld(y), _prow(coefs, 2), _prow(coefs, 3), _prow(coefs, 0), _prow(coefs, 1), _p(sums), dt(x), B, H, W, Cc,
         _stream(), nbytes=x.numel() * x.element_size() * 4.25)
    return sums


def bn_relu_bwd(gz, y, coefs, training, dgamma=None, dbeta=None, sums=None, peer=None):
    """Returns (gy, dgamma, dbeta) for z = relu(bn(y)); `dgamma` / `dbeta`: optional fp32 [C] destinations; `sums`:
    the fp64 [2, C] reduction when the kernel that produced gz already made it (gconv_dgrad_bnbwd); `peer`: the
    ddp.BNPeerGroup of a synchronised BatchNorm (its coefficients then come from the sums of every rank)."""
    B, Cc, H, W = y.shape
    dev = y.device
    es = y.element_size()
    L = lib()
    if sums is None:
        sums = torch.zeros((2, Cc), dtype=torch.float64, device=dev)
        _run("bn_relu_bwd_reduce", L.unetb200_bn_relu_bwd_reduce, _p(gz), nhwc_ld(gz), _p(y), nhwc_ld(y), _prow(coefs, 2),
             _prow(coefs, 3), _prow(coefs, 0), _prow(coefs, 1), _p(sums), dt(y), B, H, W, Cc, _stream(),
             nbytes=2.0 * y.numel() * es)
    if dgamma is None:
        dgamma = torch.empty(Cc, dtype=torch.float32, device=dev)
    if dbeta is None:
        dbeta = torch.empty(Cc, dtype=torch.float32, device=dev)
    coef = torch.empty((2, Cc), dtype=torch.float32, device=dev)
    if peer is not None:
        bn_sync_bwd_finalize(peer, sums, B * H * W, dgamma, dbeta, coef)
    else:
        _run("bn_bwd_finalize", L.unetb200_bn_bwd_finalize, _p(sums), B * H * W, 1 if training else 0, _p(dgamma),
             _p(dbeta), _p(coef), Cc, _stream())
    gy = empty_nhwc(B, Cc, H, W, y.dtype, dev)
    _run("bn_relu_bwd_apply", L.unetb200_bn_relu_bwd_apply, _p(gz), nhwc_ld(gz), _p(y), nhwc_ld(y), _prow(coefs, 2),
         _prow(coefs, 3), _prow(coefs, 0), _prow(coefs, 1), _p(coef), _p(gy), nhwc_ld(gy), dt(y), B, H, W, Cc, _stream(),
         nbytes=3.0 * y.numel() * es)
    return gy, dgamma, dbeta


def upsample2x_fwd(x, y, off):
    B, Cc, h, w = x.shape
    _run("upsample2x_fwd", lib().unetb200_upsample2x_fwd, _p(x), nhwc_ld(x), _p(y), nhwc_ld(y), dt(x), B, h, w, Cc,
         y.shape[2], y.shape[3], off[0], off[1], _stream(), nbytes=5.0 * x.numel() * x.element_size())


def upsample2x_bwd(gy, gx, off):
    B, Cc, h, w = gx.shape
    _run("upsample2x_bwd", lib().unetb200_upsample2x_bwd, _p(gy), nhwc_ld(gy), _p(gx), nhwc_ld(gx), dt(gx), B, h, w,
         Cc, gy.shape[2], gy.shape[3], off[0], off[1], _stream(), nbytes=5.0 * gx.numel() * gx.element_size())


# ------------------------------------------------------------------------------------------------
# SpatialAttention gate (UNet_SA)
# ------------------------------------------------------------------------------------------------
def sa_forward(x, w, out):
    """out = x * sigmoid(conv7x7([mean_c x, max_c x])); returns the fp32 maps (stats [B,H,W,2], gate [B,H,W])."""
    B, Cc, H, W = x.shape
    stats = torch.empty((B, H, W, 2), dtype=torch.float32, device=x.device)
    gate = torch.empty((B, H, W), dtype=torch.float32, device=x.device)
    _run("sa_forward", lib().unetb200_sa_forward, _p(x), nhwc_ld(x), _p(w), _p(stats), _p(gate), _p(out), nhwc_ld(out),
         dt(x), B, H, W, Cc, _stream(), kernels=3, nbytes=3.0 * x.numel() * x.element_size())
    return stats, gate


def sa_backward(g, x, w, stats, gate, dx, dw):
    B, Cc, H, W = x.shape
    ws = torch.empty(lib().unetb200_sa_backward_workspace(B, H, W), dtype=torch.float32, device=x.device)
    _run("sa_backward", lib().unetb200_sa_backward, _p(g), nhwc_ld(g), _p(x), nhwc_ld(x), _p(w), _p(stats), _p(gate),
         _p(dx), nhwc_ld(dx), _p(dw), _p(ws), dt(x), B, H, W, Cc, _stream(), kernels=5,
         nbytes=5.0 * x.numel() * x.element_size())


# ------------------------------------------------------------------------------------------------
# OutConv
# ------------------------------------------------------------------------------------------------
def outconv_fwd(x, w, bias, logits):
    B, Cc, H, W = x.shape
    K = w.shape[0]
    _run("outconv_fwd", lib().unetb200_outconv_fwd, _p(x), nhwc_ld(x), _p(w), _p(bias), _p(logits), dt(x), B * H * W,
         Cc, K, _stream(), nbytes=(x.numel() + logits.numel()) * x.element_size())


# OutConv backward fused with the BatchNorm-backward reduction of the stage below: measured at B = 16, 512x512, 64
# channels, 2 classes: 0.786 ms against 0.380 ms + 0.23 ms for the separate reduction pass (the 48 extra registers
# halve the occupancy of this latency-bound stream), so the fused form is opt-in; it stays tested.
OUTCONV_FUSE = os.environ.get("UNETB200_OUTCONV_FUSE", "0") != "0"


def outconv_bwd(x, w, glogits, gx, dw, dbias, below=None):
    """`below` = (yprev, coefs) of the conv-BN-ReLU stage whose activation is x: when the fused kernel covers the
    shape the BatchNorm-backward reduction of that stage is made here (gx is its output gradient) and returned as
    fp64 sums[2, C]; else None."""
    B, Cc, H, W = x.shape
    K = w.shape[0]
    n = lib().unetb200_outconv_bwd_workspace(B * H * W, Cc, K)
    ws = torch.empty(n, dtype=torch.float32, device=x.device)
    if below is not None and gx is not None and OUTCONV_FUSE:
        yprev, coefs = below
        if coefs.is_contiguous() and lib().unetb200_outconv_bwd_bnbwd_supported(
                _p(x), nhwc_ld(x), _p(gx), nhwc_ld(gx), _p(yprev), nhwc_ld(yprev), dt(x), Cc, K):
            sums = torch.zeros((2, Cc), dtype=torch.float64, device=x.device)
            _run("outconv_bwd", lib().unetb200_outconv_bwd_bnbwd, _p(x), nhwc_ld(x), _p(w), _p(glogits), _p(gx),
                 nhwc_ld(gx), _p(dw), _p(dbias), _p(ws), _p(yprev), nhwc_ld(yprev), _p(coefs), _p(sums), dt(x),
                 B * H * W, Cc, K, _stream(), kernels=2, nbytes=(3 * x.numel() + glogits.numel()) * x.element_size())
            return sums
    _run("outconv_bwd", lib().unetb200_outconv_bwd, _p(x), nhwc_ld(x), _p(w), _p(glogits), _p(gx),
         nhwc_ld(gx) if gx is not None else 0, _p(dw), _p(dbias), _p(ws), dt(x), B * H * W, Cc, K, _stream(),
         kernels=2, nbytes=(2 * x.numel() + glogits.numel()) * x.element_size())
    return None
