"""Kernel ledger: every instantiation of the convolution engines and OutConv (conv_tc2/3/4.cu, conv_halo*.cu,
conv_narrow.cu, conv_first*.cu, conv_simt*.cu, outconv.cu) against a CPU float64 reference, and the kernels each case
ran, read from a torch.profiler trace.

A case is one C-ABI operation (fprop + BatchNorm statistics, dgrad, wgrad with its split reduction, a fused
epilogue, ConvTranspose, OutConv, a weight pack) on seeded operands.  Running a case

* records the in-scope kernels it launched and requires them to be exactly the ledger's set for it: a route or
  support predicate that moves a case to another kernel fails and names the kernel;
* compares every output with the fp64 reference of the same operation on the operands rounded to the device dtype,
  element by element:  |dev - ref| <= a * u_out * |ref| + b * (u_op + K * 2^-24) * A, where A is the same reduction
  over absolute values (|x| (*) |w|; sum |x||gy| for wgrad; sum |y| and sum y^2 for statistics) and K its length;
* checks sentinel guard bands around every output (the untouched channels of a slice destination and the borders of
  a padded ConvTranspose destination included), that the inputs are byte-identical afterwards, and that a second run
  gives bit-equal outputs -- apart from the outputs reduced with float atomics, held to 1e-6 relative: statistics
  that went through stats_reduce_kernel (conv_simt.cu, which also finishes conv_first.cu's), and OutConv dW / db of
  the scalar backward kernel (outconv.cu).

`python tests/kernel_ledger.py --set NAME --out FILE` runs the cases of one switch set in a process of its own (the
switches are read once into statics) and writes the per-case results as JSON.
"""
import argparse
import json
import math
import os
import sys

import torch
import torch.nn.functional as F

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
PKG = os.path.join(ROOT, "unet-medical-image-contour-segmentation_b200")
for _p in (PKG, ROOT):
    if _p not in sys.path:
        sys.path.insert(0, _p)

DEV = "cuda"
BF, FP = torch.bfloat16, torch.float32
SENT = 3.0           # guard-band sentinel
GUARD = 4096         # guard elements either side of every output

# ------------------------------------------------------------------------------------------------
# the comparator (also used without a GPU by tests/test_kernel_ledger_cpu.py)
# ------------------------------------------------------------------------------------------------
# u_out: unit roundoff of the stored output; u_op: operand rounding inside the product (TF32 operands: 2^-10 for the
# product of two operands each rounded to 10 mantissa bits; the fused OutConv head multiplies its bf16-rounded
# activation).  a and b are fixed once per compute type (a <= 2, b <= 4); no case sets its own.
COMPUTE = {
    "bf16": dict(u_out=2.0 ** -8, u_op=0.0),
    "bf16_head": dict(u_out=2.0 ** -8, u_op=2.0 ** -8),
    "fp32": dict(u_out=0.0, u_op=0.0),
    "tf32": dict(u_out=0.0, u_op=2.0 ** -10),
    "acc32": dict(u_out=0.0, u_op=0.0),      # fp32 outputs of a bf16 / fp32 product (wgrad, statistics, dW)
}
A_COEF, B_COEF = 2.0, 4.0


def bound(ref, A, K, compute):
    c = COMPUTE[compute]
    return A_COEF * c["u_out"] * ref.abs() + B_COEF * (c["u_op"] + K * 2.0 ** -24) * A


def err_over_bound(dev, ref, A, K, compute):
    """worst |dev - ref| / bound over the elements (inf where a NaN or a missed store shows)"""
    dev = dev.double()
    bd = bound(ref, A, K, compute)
    e = (dev - ref).abs()
    bad = ~torch.isfinite(e)
    r = torch.where(bd > 0, e / bd.clamp_min(1e-300), torch.where(e > 0, torch.full_like(e, math.inf), torch.zeros_like(e)))
    r = torch.where(bad, torch.full_like(r, math.inf), r)
    return float(r.max()) if r.numel() else 0.0


def rel(dev, ref):
    """the suite's older max-abs metric: max |dev - ref| / max |ref|"""
    dev, ref = dev.double(), ref.double()
    d = (dev - ref).abs().max().item()
    return d / max(ref.abs().max().item(), 1e-30)


REL_TOL = {"bf16": 1.2e-2, "bf16_head": 1.2e-2, "tf32": 2e-3, "fp32": 2e-5, "acc32": 5e-3}


# ---- fp64 references (NCHW, CPU) --------------------------------------------------------------
def ref_conv3x3(x, w):
    x, w = x.double(), w.double()
    return F.conv2d(x, w, padding=1), F.conv2d(x.abs(), w.abs(), padding=1)


def ref_dgrad3x3(gy, w):
    wt = w.double().flip(2, 3).transpose(0, 1)
    return F.conv2d(gy.double(), wt, padding=1), F.conv2d(gy.double().abs(), wt.abs(), padding=1)


def ref_wgrad3x3(x, gy):
    x, gy = x.double(), gy.double()
    sh = (gy.shape[1], x.shape[1], 3, 3)
    return (torch.nn.grad.conv2d_weight(x, sh, gy, padding=1),
            torch.nn.grad.conv2d_weight(x.abs(), sh, gy.abs(), padding=1))


def ref_convT(x, w, b):
    x, w, b = x.double(), w.double(), b.double()
    return F.conv_transpose2d(x, w, b, stride=2), F.conv_transpose2d(x.abs(), w.abs(), b.abs(), stride=2)


def ref_convT_dgrad(gy, w):
    gy, w = gy.double(), w.double()
    return F.conv2d(gy, w, stride=2), F.conv2d(gy.abs(), w.abs(), stride=2)


def ref_convT_wgrad(x, gy):
    x, gy = x.double(), gy.double()
    B, Co, H, W = gy.shape
    g6 = gy.reshape(B, Co, H // 2, 2, W // 2, 2)
    return (torch.einsum("bcij,boikjl->cokl", x, g6), torch.einsum("bcij,boikjl->cokl", x.abs(), g6.abs()))


def ref_stats(y):
    """BatchNorm statistics of the stored output: sums over (B, H, W) of y and y^2; A = sum |y|, sum y^2"""
    y = y.double()
    s = torch.stack([y.sum((0, 2, 3)), (y * y).sum((0, 2, 3))])
    return s, torch.stack([y.abs().sum((0, 2, 3)), (y * y).sum((0, 2, 3))])


def ref_outconv(x, w, b):
    """x [B,C,H,W], w [K,C] -> logits [B,K,H,W]"""
    x, w = x.double(), w.double()
    y = torch.einsum("bchw,kc->bkhw", x, w)
    A = torch.einsum("bchw,kc->bkhw", x.abs(), w.abs())
    if b is not None:
        y = y + b.double().view(1, -1, 1, 1)
        A = A + b.double().abs().view(1, -1, 1, 1)
    return y, A


def ref_bnbwd_sums(gx, y, coefs):
    """sums[2, C] of the BatchNorm + ReLU backward of the layer with raw output y, gx the gradient of relu(bn(y)):
    [sum g*m, sum g*m*(y-mean)*invstd], m = (y*scale + shift > 0) evaluated as the kernels do (one fp32 fma)"""
    c = coefs.double()
    v = lambda t: t.view(1, -1, 1, 1)  # noqa: E731
    m = (torch.addcmul(v(coefs[3]).float(), y.float(), v(coefs[2]).float()) > 0).double()
    g = gx.double() * m
    xh = (y.double() - v(c[0])) * v(c[1])
    s = torch.stack([g.sum((0, 2, 3)), (g * xh).sum((0, 2, 3))])
    A = torch.stack([g.abs().sum((0, 2, 3)), (g * xh).abs().sum((0, 2, 3))])
    return s, A


def rq(x, dtype):
    return x.detach().to(dtype).float()


# ------------------------------------------------------------------------------------------------
# which kernel ran
# ------------------------------------------------------------------------------------------------
SCOPE_BASES = frozenset("""
first_conv_fprop_kernel first_conv_fprop_px4_kernel first_conv_fprop_tiled_kernel first_conv_wgrad_kernel
first_conv_wgrad_tiled_kernel first_narrow_fprop_kernel first_narrow_wgrad_kernel first_tc_kernel fprop_narrow_f32_kernel
gconv_fprop_simt_kernel gconv_wgrad_simt_kernel halo_conv_kernel halo_t_dgrad_kernel halo_t_fprop_kernel
halo_t_wgrad_kernel halo_wgrad_kernel narrow_conv_kernel narrow_wgrad_kernel outconv_bwd_scalar_kernel
outconv_bwd_vec_kernel outconv_fwd_scalar_kernel outconv_fwd_vec_kernel outconv_reduce_kernel pack_multi_kernel
pack_weights_kernel pack_weights_t_kernel stats_reduce_kernel tc2_fprop_kernel tc2_stats_reduce_kernel tc2_wgrad_kernel
tc3_conv_kernel tc3_stats_reduce_kernel tc3_wgrad_kernel tc4_wgrad_kernel wgrad_narrow_f32_kernel wgrad_reduce_kernel
wgrad_reduce_multi_kernel wgrad_reduce_t4_kernel wgrad_reduce_t_kernel""".split())

# the memory-bound kernels of the library (elementwise, loss, io_tail, bn_sync, attention, optim): not in the ledger,
# but named, so that a kernel of a new kind has to be put on one side or the other
OUT_OF_SCOPE_BASES = frozenset("""
add_channels_kernel bce_dice_bwd_kernel bce_dice_finalize_kernel bce_dice_fwd_kernel bn_bwd_finalize_kernel
bn_eval_coeffs_kernel bn_finalize_kernel bn_relu_apply_kernel bn_relu_apply_pool_kernel bn_relu_bwd_apply_kernel
bn_relu_bwd_reduce_kernel bn_sync_bwd_finalize_kernel bn_sync_finalize_kernel boundary_counts_kernel
boundary_finalize_kernel ce_dice_bwd_kernel ce_dice_finalize_kernel ce_dice_fwd_kernel channel_sum_kernel
channel_sum_vec_kernel convert_flat_kernel copy_channels_kernel dice_bwd_kernel dice_finalize_kernel dice_fwd_kernel
double_to_float_kernel eval_counts_kernel eval_counts_packed_kernel eval_dice_finalize_kernel gather_nhwc_kernel
grad_sqnorm_amp_kernel grad_sqnorm_kernel maxpool2_bwd_bnreduce_kernel maxpool2_bwd_kernel maxpool2_fwd_kernel
resize_argmax_kernel rmsprop_step_amp_kernel rmsprop_step_kernel rot_convert_kernel sa_apply_kernel sa_bwd_dgate_kernel
sa_bwd_dstats_kernel sa_bwd_dw_kernel sa_bwd_dw_reduce_kernel sa_bwd_dx_kernel sa_gate_tiled_kernel sa_stats_kernel
sa_stats_scalar_kernel split_tf32_kernel u8_any_gt1_kernel upsample2x_bwd_kernel upsample2x_fwd_kernel
zero_channels_kernel""".split())


def normalise(name):
    """'void ub::(anonymous namespace)::tc3_conv_kernel<__nv_bfloat16, 64, ...>(ub::Tc3Params)' ->
    'tc3_conv_kernel<__nv_bfloat16, 64, ...>'"""
    n = name.strip()
    if n.startswith("void "):
        n = n[5:]
    n = n.replace("(anonymous namespace)::", "").replace("ub::", "")
    depth = 0
    for i, ch in enumerate(n):
        if ch == "<":
            depth += 1
        elif ch == ">":
            depth -= 1
        elif ch == "(" and depth == 0:
            return n[:i].strip()
    return n


def base(name):
    return name.split("<", 1)[0]


def in_scope(name):
    return base(name) in SCOPE_BASES


# ------------------------------------------------------------------------------------------------
# device plumbing (imported lazily: the CPU tests use only the part above)
# ------------------------------------------------------------------------------------------------
def _dev():
    from unetb200 import _lib, backward_pass, ops  # noqa: F401
    from unetb200 import functional as UF
    return _lib, ops, UF, backward_pass


class Guarded:
    """An output of `size` / `stride` at element `offset` of a flat buffer whose every other element (guard bands,
    channels outside a slice, borders of a padded destination) holds SENT; the output itself starts as `init` (NaN:
    a missed store shows as a failed comparison)."""

    def __init__(self, numel, dtype, size, stride, offset=0, init=float("nan")):
        self.flat = torch.full((2 * GUARD + numel,), SENT, dtype=dtype, device=DEV)
        self.view = self.flat.as_strided(size, stride, GUARD + offset)
        self.view.fill_(init)

    def ptr(self, offset=0):
        return self.flat.data_ptr() + (GUARD + offset) * self.flat.element_size()

    def intact(self):
        c = self.flat.clone()
        c.as_strided(self.view.size(), self.view.stride(), self.view.storage_offset()).fill_(SENT)
        return bool((c == SENT).all())


def g_nhwc(B, C, H, W, dtype, ld=None, c0=0, init=float("nan")):
    ld = ld or C
    return Guarded(B * H * W * ld, dtype, (B, C, H, W), (H * W * ld, 1, W * ld, ld), c0, init)


def g_vec(shape, dtype, init=float("nan"), stride=None):
    n = 1
    for s in shape:
        n *= s
    if stride is None:
        stride, acc = [], 1
        for s in reversed(shape):
            stride.insert(0, acc)
            acc *= s
    return Guarded(n, dtype, tuple(shape), tuple(stride), 0, init)


def d_nhwc(x, dtype, ld=None, c0=0, seed=0):
    """device NHWC copy of CPU NCHW x; with ld > C the other channels of the pixel hold junk (a slice input)"""
    B, C, H, W = x.shape
    ld = ld or C
    g = torch.Generator().manual_seed(seed + 7)
    buf = (torch.randn(B, H, W, ld, generator=g) * 50).to(dtype).to(DEV)
    v = buf.as_strided((B, C, H, W), (H * W * ld, 1, W * ld, ld), c0)
    v.copy_(x.to(DEV).to(dtype))
    return buf, v


def _bits(t):
    t = t.detach().contiguous().view(-1)
    return t.view({1: torch.uint8, 2: torch.int16, 4: torch.int32, 8: torch.int64}[t.element_size()])


STATS_ATOMIC = frozenset({"stats_reduce_kernel"})
OUTCONV_ATOMIC = frozenset({"outconv_bwd_scalar_kernel"})


class Out:
    """one compared output: guarded device buffer, fp64 reference, A, K, compute type; `atomic`: the kernels (base
    names) whose presence means the output was reduced with float atomics"""

    def __init__(self, name, g, ref=None, A=None, K=1, compute="bf16", atomic=frozenset(), exact_of=None):
        self.name, self.g, self.ref, self.A, self.K, self.compute, self.atomic = name, g, ref, A, K, compute, atomic
        self.exact_of = exact_of      # callable(view) -> expected tensor, compared exactly (pooled = maxpool(z))


class Case:
    def __init__(self, cid, prepare, env="default"):
        self.id = cid if env == "default" else f"{env}/{cid}"
        self.prepare, self.env = prepare, env


def launched_kernels(fn):
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        r = fn()
        torch.cuda.synchronize()
    names = sorted({normalise(ev.name) for ev in prof.events() if ev.device_type == torch.autograd.DeviceType.CUDA})
    return r, names


def run_case(case):
    """-> dict(kernels, worst, rel, failures)"""
    inputs, launch = case.prepare()
    before = [i.clone() for i in inputs]
    outs1, names = launched_kernels(launch)
    outs2 = launch()
    torch.cuda.synchronize()
    fails, worst, wrel = [], 0.0, 0.0
    for a, b in zip(before, inputs):
        if not torch.equal(_bits(a), _bits(b)):
            fails.append("input changed")
    for o1, o2 in zip(outs1, outs2):
        for o in (o1, o2):
            if not o.g.intact():
                fails.append(f"{o.name}: guard band / untouched region changed")
        v1, v2 = o1.g.view, o2.g.view
        if any(base(n) in o1.atomic for n in names):
            d = (v1.double() - v2.double()).abs().max().item() if v1.numel() else 0.0
            if not d <= 1e-6 * max(v1.double().abs().max().item(), 1e-30):
                fails.append(f"{o1.name}: runs differ by {d:.3e} (atomics: 1e-6 relative)")
        elif not torch.equal(_bits(v1), _bits(v2)):
            fails.append(f"{o1.name}: second run not bit-equal")
        if o1.exact_of is not None:
            if not torch.equal(o1.exact_of().float().cpu(), v1.float().cpu()):
                fails.append(f"{o1.name}: not the exact function of the stored output")
        if o1.ref is not None:
            dv = v1.detach().double().cpu()
            e = err_over_bound(dv, o1.ref, o1.A, o1.K, o1.compute)
            r = rel(dv, o1.ref)
            worst, wrel = max(worst, e), max(wrel, r)
            if not e <= 1.0:
                fails.append(f"{o1.name}: err/bound {e:.3g} (rel {r:.3g})")
    in_sc = [n for n in names if in_scope(n)]
    return dict(kernels=in_sc, worst=worst, rel=wrel, failures=fails)


# ------------------------------------------------------------------------------------------------
# case builders
# ------------------------------------------------------------------------------------------------
def _gen(seed):
    return torch.Generator().manual_seed(seed)


def _cname(dt):
    return "bf16" if dt == BF else "fp32"


def _compute(dt, algo_tc):
    return "bf16" if dt == BF else ("tf32" if algo_tc else "fp32")


def _desc3(ops, dt, algo, B, H, W, Cin, ld_in, N, ld_out):
    d = ops.make_gconv(ops._DT[dt], algo, B, H, W, Cin, ops.TAPS3, 1, (0, 0), H, W, ld_in, N, 1, 1, (0, 0), H, W, ld_out)
    d.algo = algo
    return d


def _algo(lib, name):
    return {"tc": lib.ALGO_TC, "auto": lib.ALGO_AUTO, "simt": lib.ALGO_SIMT, "prefer": lib.ALGO_PREFER_TC}[name]


def _tf32(dt, algo):
    return dt == FP and algo in ("tc", "prefer")


def conv3x3_fprop(dt, algo, B, Ci, Co, H, W, seed, ld_in=None, c0_in=0, ld_out=None, c0_out=0, stats=True, bias=False):
    def prepare():
        lib, ops, UF, _ = _dev()
        g = _gen(seed)
        x = rq(torch.randn(B, Ci, H, W, generator=g), dt)
        w = torch.randn(Co, Ci, 3, 3, generator=g) / (3 * Ci ** 0.5)
        ref, A = ref_conv3x3(x, rq(w, dt))
        b = torch.randn(Co, generator=g) if bias else None
        if bias:
            bq = rq(b, dt).double().view(1, -1, 1, 1)      # added in the storage dtype, as for ConvTranspose
            ref, A = ref + bq, A + bq.abs()
        bd = b.to(DEV) if bias else None
        xb, xv = d_nhwc(x, dt, ld_in, c0_in, seed)
        wp = UF.pack3x3_fprop(w.to(DEV), dt)
        a = _algo(lib, algo)
        comp = _compute(dt, _tf32(dt, algo))

        def launch():
            y = g_nhwc(B, Co, H, W, dt, ld_out, c0_out)
            st = g_vec((2 * Co,), torch.float64, init=0.0) if stats else None
            d = _desc3(ops, dt, a, B, H, W, Ci, ld_in or Ci, Co, ld_out or Co)
            ops.gconv_fprop(d, xv, wp, bd, y.view, st.view if st is not None else None)
            outs = [Out("y", y, ref, A, 9 * Ci + bias, comp)]
            if stats:
                torch.cuda.synchronize()
                sref, sA = ref_stats(y.view.detach().double().cpu())
                outs.append(Out("stats", st, sref.reshape(-1), sA.reshape(-1), B * H * W, "acc32", atomic=STATS_ATOMIC))
            return outs
        return [xb, wp] + ([bd] if bias else []), launch
    return prepare


def conv3x3_dgrad(dt, algo, B, Ci, Co, H, W, seed, ld_out=None, c0_out=0):
    """data gradient (Co -> Ci channels): the fprop kernels on the rotated, transposed weights"""
    def prepare():
        lib, ops, UF, _ = _dev()
        g = _gen(seed)
        gy = rq(torch.randn(B, Co, H, W, generator=g), dt)
        w = torch.randn(Co, Ci, 3, 3, generator=g) / (3 * Co ** 0.5)
        ref, A = ref_dgrad3x3(gy, rq(w, dt))
        gb, gv = d_nhwc(gy, dt, seed=seed)
        wp = UF.pack3x3_dgrad(w.to(DEV), dt)
        a = _algo(lib, algo)
        comp = _compute(dt, _tf32(dt, algo))

        def launch():
            gx = g_nhwc(B, Ci, H, W, dt, ld_out, c0_out)
            d = _desc3(ops, dt, a, B, H, W, Co, Co, Ci, ld_out or Ci)
            ops.gconv_fprop(d, gv, wp, None, gx.view, None, kind="dgrad")
            return [Out("gx", gx, ref, A, 9 * Co, comp)]
        return [gb, wp], launch
    return prepare


def _wgrad_call(lib, ops, bp, d, x, gy, dst, st, sc, sq, sn, multi):
    """plan, split kernel into guarded partials, split reduction into the guarded parameter-layout dst"""
    import ctypes as C
    splits, used = C.c_int(0), C.c_int(0)
    L = ops.lib()
    lib.check(L.unetb200_gconv_wgrad_plan(C.byref(d), C.byref(splits), C.byref(used)), "gconv_wgrad_plan")
    K = d.ntaps * d.Cin
    parts = g_vec((splits.value * K * d.N,), torch.float32)
    d2 = lib.GConv.from_buffer_copy(d)
    d2.algo = used.value
    lib.check(L.unetb200_gconv_wgrad(C.byref(d2), ops._p(x), ops._p(gy), C.c_void_p(parts.ptr()), splits.value,
                                     ops._stream()), "gconv_wgrad")
    Cq = d.N // d.nquad
    if multi:
        bp._reduce_multi([(parts.view, dst.ptr(), st, sc, sq, sn, splits.value, d.ntaps, d.Cin, d.N, Cq)])
    else:
        lib.check(L.unetb200_wgrad_reduce(C.c_void_p(parts.ptr()), splits.value, d.ntaps, d.Cin, d.N, Cq,
                                          C.c_void_p(dst.ptr()), st, sc, sq, sn, 0, ops._stream()), "wgrad_reduce")
    return parts


def conv3x3_wgrad(dt, algo, B, Ci, Co, H, W, seed, layout="oihw", ld_in=None, c0_in=0):
    """weight gradient after the split reduction, in the parameter layout: 'oihw' (contiguous), 'cl' (channels_last)
    or 'multi' (contiguous, through the batched reduction the backward pass defers to)"""
    def prepare():
        lib, ops, UF, bp = _dev()
        g = _gen(seed)
        x = rq(torch.randn(B, Ci, H, W, generator=g), dt)
        gy = rq(torch.randn(B, Co, H, W, generator=g), dt)
        ref, A = ref_wgrad3x3(x, gy)
        xb, xv = d_nhwc(x, dt, ld_in, c0_in, seed)
        gb, gv = d_nhwc(gy, dt, seed=seed + 1)
        a = _algo(lib, algo)

        def launch():
            if layout == "cl":
                dst = g_vec((Co, Ci, 3, 3), torch.float32, stride=(9 * Ci, 1, 3 * Ci, Ci))
                st, sc, sn = Ci, 1, 9 * Ci
            else:
                dst = g_vec((Co, Ci, 3, 3), torch.float32)
                st, sc, sn = 1, 9, 9 * Ci
            d = _desc3(ops, dt, a, B, H, W, Ci, ld_in or Ci, Co, Co)
            parts = _wgrad_call(lib, ops, bp, d, xv, gv, dst, st, sc, 0, sn, layout == "multi")
            return [Out("dW", dst, ref, A, B * H * W, "tf32" if _tf32(dt, algo) else "acc32"), Out("partials", parts)]
        return [xb, gb], launch
    return prepare


def _affine_coefs(g, C):
    mean, invstd = torch.randn(C, generator=g) * 0.2, torch.rand(C, generator=g) + 0.5
    scale = (torch.rand(C, generator=g) + 0.5) * invstd
    shift = torch.randn(C, generator=g) * 0.3 - mean * scale
    return torch.stack([mean, invstd, scale, shift]).contiguous()


def conv3x3_affine(dt, algo, B, Ci, Co, H, W, seed, pool=False, ld_out=None, c0_out=0):
    """inference epilogue: z = relu(conv * scale + shift) (and MaxPool2d(2) of z as a second output)"""
    def prepare():
        lib, ops, UF, _ = _dev()
        g = _gen(seed)
        x = rq(torch.randn(B, Ci, H, W, generator=g), dt)
        w = torch.randn(Co, Ci, 3, 3, generator=g) * (2.0 / (9 * Ci)) ** 0.5
        coefs = _affine_coefs(g, Co)
        y, A = ref_conv3x3(x, rq(w, dt))
        sc, sh = coefs[2].double().view(1, -1, 1, 1), coefs[3].double().view(1, -1, 1, 1)
        ref = torch.relu(y * sc + sh)
        Az = A * sc.abs() + sh.abs()
        xb, xv = d_nhwc(x, dt, seed=seed)
        wp = UF.pack3x3_fprop(w.to(DEV), dt)
        cd = coefs.to(DEV)
        a = _algo(lib, algo)
        comp = _compute(dt, _tf32(dt, algo))

        def launch():
            z = g_nhwc(B, Co, H, W, dt, ld_out, c0_out)
            d = _desc3(ops, dt, a, B, H, W, Ci, Ci, Co, ld_out or Co)
            outs = [Out("z", z, ref, Az, 9 * Ci, comp)]
            if pool:
                p = g_nhwc(B, Co, H // 2, W // 2, dt)
                assert ops.gconv_fprop_affine_relu_pool_supported(d, xv, wp, z.view, p.view), "pool fold not supported"
                ops.gconv_fprop_affine_relu(d, xv, wp, cd, z.view, p.view)
                outs.append(Out("pooled", p, F.max_pool2d(ref, 2), F.max_pool2d(Az, 2), 9 * Ci, comp,
                                exact_of=lambda: F.max_pool2d(z.view.float(), 2)))
            else:
                assert ops.gconv_fprop_affine_relu_supported(d, xv, wp, z.view), "affine fold not supported"
                ops.gconv_fprop_affine_relu(d, xv, wp, cd, z.view)
            return outs
        return [xb, wp, cd], launch
    return prepare


def conv3x3_head(B, Ci, H, W, ncls, seed, bias=True):
    """last conv of the network in inference: conv3x3 (-> 64) -> BatchNorm(eval) -> ReLU -> OutConv 1x1 in one kernel"""
    Co = 64

    def prepare():
        lib, ops, UF, _ = _dev()
        g = _gen(seed)
        x = rq(torch.randn(B, Ci, H, W, generator=g), BF)
        w = torch.randn(Co, Ci, 3, 3, generator=g) * (2.0 / (9 * Ci)) ** 0.5
        coefs = _affine_coefs(g, Co)
        ow = torch.randn(ncls, Co, generator=g) * 0.3
        ob = torch.randn(ncls, generator=g) if bias else None
        y, A = ref_conv3x3(x, rq(w, BF))
        sc, sh = coefs[2].double().view(1, -1, 1, 1), coefs[3].double().view(1, -1, 1, 1)
        z = torch.relu(y * sc + sh)
        ref, Ah = ref_outconv(z, rq(ow, BF), rq(ob, BF) if bias else None)
        # A of the head: |w_oc| (*) (scale-weighted conv A + |shift|) -- the activation's own error propagates too
        Ah = torch.einsum("bchw,kc->bkhw", A * sc.abs() + sh.abs(), rq(ow, BF).double().abs()) + \
            (rq(ob, BF).double().abs().view(1, -1, 1, 1) if bias else 0.0)
        xb, xv = d_nhwc(x, BF, seed=seed)
        wp = UF.pack3x3_fprop(w.to(DEV), BF)
        cd, owd = coefs.to(DEV), ow.to(DEV)
        obd = ob.to(DEV) if bias else None
        a = lib.ALGO_TC

        def launch():
            lg = g_vec((B, H, W, ncls), BF)
            d = _desc3(ops, BF, a, B, H, W, Ci, Ci, Co, Co)
            assert ops.gconv_fprop_affine_relu_outconv_supported(d, xv, wp, ncls), "fused head not supported"
            ops.gconv_fprop_affine_relu_outconv(d, xv, wp, cd, owd, obd, lg.view)
            return [Out("logits", lg, ref.permute(0, 2, 3, 1), Ah.permute(0, 2, 3, 1), 9 * Ci + Co, "bf16_head")]
        ins = [xb, wp, cd, owd] + ([obd] if bias else [])
        return ins, launch
    return prepare


def conv3x3_bnbwd(dt, algo, B, Ci, Co, H, W, seed, ld_y=None):
    """dgrad (Co -> Ci) with the BatchNorm + ReLU backward reduction of the layer below in the epilogue"""
    def prepare():
        import ctypes as C
        lib, ops, UF, _ = _dev()
        g = _gen(seed)
        gy = rq(torch.randn(B, Co, H, W, generator=g), dt)
        w = torch.randn(Co, Ci, 3, 3, generator=g) / (3 * Co ** 0.5)
        yprev = rq(torch.randn(B, Ci, H, W, generator=g), dt)
        coefs = _affine_coefs(g, Ci)
        ref, A = ref_dgrad3x3(gy, rq(w, dt))
        gb, gv = d_nhwc(gy, dt, seed=seed)
        yb, yv = d_nhwc(yprev, dt, ld_y, 0, seed + 3)
        wp = UF.pack3x3_dgrad(w.to(DEV), dt)
        cd = coefs.to(DEV)
        a = _algo(lib, algo)
        comp = _compute(dt, _tf32(dt, algo))

        def launch():
            gx = g_nhwc(B, Ci, H, W, dt)
            sums = g_vec((2, Ci), torch.float64, init=0.0)
            d = _desc3(ops, dt, a, B, H, W, Co, Co, Ci, Ci)
            assert ops.gconv_dgrad_bnbwd_supported(d, gv, wp, gx.view), "dgrad + BatchNorm backward not supported"
            L = ops.lib()
            ws = torch.empty(L.unetb200_gconv_stats_workspace(C.byref(d)), dtype=torch.float32, device=DEV)
            lib.check(L.unetb200_gconv_dgrad_bnbwd(C.byref(d), ops._p(gv), ops._p(wp), ops._p(gx.view), ops._p(yv),
                                                   ops.nhwc_ld(yv), ops._p(cd), C.c_void_p(sums.ptr()), ops._p(ws),
                                                   ops._stream()), "gconv_dgrad_bnbwd")
            torch.cuda.synchronize()
            sref, sA = ref_bnbwd_sums(gx.view.detach().double().cpu(), yprev, coefs)
            return [Out("gx", gx, ref, A, 9 * Co, comp),
                    Out("sums", sums, sref, sA, B * H * W, "acc32", atomic=STATS_ATOMIC)]
        return [gb, yb, wp, cd], launch
    return prepare


def convT_fprop(dt, algo, B, Ci, Co, h, w_, seed, pad=(0, 0)):
    """ConvTranspose2d(k=2, s=2) + bias into the second channel half of a concat buffer, at the centring offset of
    a padded destination (the border and the skip half stay untouched)"""
    def prepare():
        lib, ops, UF, _ = _dev()
        g = _gen(seed)
        x = rq(torch.randn(B, Ci, h, w_, generator=g), dt)
        w = torch.randn(Ci, Co, 2, 2, generator=g) / (Ci ** 0.5)
        b = torch.randn(Co, generator=g)
        ref, A = ref_convT(x, rq(w, dt), rq(b, dt))   # every engine adds the bias in the storage dtype
        H, W = 2 * h + pad[0], 2 * w_ + pad[1]
        off = (pad[0] // 2, pad[1] // 2)
        xb, xv = d_nhwc(x, dt, seed=seed)
        wp = UF.packT_fprop(w.to(DEV), dt)
        bd = b.to(DEV)
        a = _algo(lib, algo)
        comp = _compute(dt, _tf32(dt, algo))

        def launch():
            ld = 2 * Co
            cat = Guarded(B * H * W * ld, dt, (B, Co, 2 * h, 2 * w_), (H * W * ld, 1, W * ld, ld),
                          Co + (off[0] * W + off[1]) * ld)
            up = cat.flat.as_strided((B, Co, H, W), (H * W * ld, 1, W * ld, ld), GUARD + Co)
            d = ops.make_gconv(ops._DT[dt], a, B, h, w_, Ci, ops.TAPS1, 1, (0, 0), h, w_, Ci, 4 * Co, 4, 2, off, H, W, ld)
            d.algo = a
            ops.gconv_fprop(d, xv, wp, bd, up, None)
            return [Out("up", cat, ref, A, Ci + 1, comp)]
        return [xb, wp, bd], launch
    return prepare


def convT_dgrad(dt, algo, B, Ci, Co, h, w_, seed, pad=(0, 0)):
    def prepare():
        lib, ops, UF, _ = _dev()
        g = _gen(seed)
        H, W = 2 * h + pad[0], 2 * w_ + pad[1]
        off = (pad[0] // 2, pad[1] // 2)
        gy = rq(torch.randn(B, Co, 2 * h, 2 * w_, generator=g), dt)
        w = torch.randn(Ci, Co, 2, 2, generator=g) / (Co ** 0.5)
        ref, A = ref_convT_dgrad(gy, rq(w, dt))
        # the gradient of the up half of the concat buffer; junk in the skip half and the border
        gfull = torch.randn(B, Co, H, W, generator=g) * 50
        gfull[:, :, off[0]:off[0] + 2 * h, off[1]:off[1] + 2 * w_] = gy
        gb, gv = d_nhwc(gfull, dt, 2 * Co, Co, seed)
        wp = UF.packT_dgrad(w.to(DEV), dt)
        a = _algo(lib, algo)
        comp = _compute(dt, _tf32(dt, algo))

        def launch():
            gx = g_nhwc(B, Ci, h, w_, dt)
            d = ops.make_gconv(ops._DT[dt], a, B, h, w_, Co, ops.TAPS_Q, 2, off, H, W, 2 * Co, Ci, 1, 1, (0, 0), h, w_, Ci)
            d.algo = a
            ops.gconv_fprop(d, gv, wp, None, gx.view, None, kind="dgrad")
            return [Out("gx", gx, ref, A, 4 * Co, comp)]
        return [gb, wp], launch
    return prepare


def convT_wgrad(dt, algo, B, Ci, Co, h, w_, seed, pad=(0, 0)):
    def prepare():
        lib, ops, UF, bp = _dev()
        g = _gen(seed)
        H, W = 2 * h + pad[0], 2 * w_ + pad[1]
        off = (pad[0] // 2, pad[1] // 2)
        x = rq(torch.randn(B, Ci, h, w_, generator=g), dt)
        gy = rq(torch.randn(B, Co, 2 * h, 2 * w_, generator=g), dt)
        ref, A = ref_convT_wgrad(x, gy)
        gfull = torch.randn(B, Co, H, W, generator=g) * 50
        gfull[:, :, off[0]:off[0] + 2 * h, off[1]:off[1] + 2 * w_] = gy
        xb, xv = d_nhwc(x, dt, seed=seed)
        gb, gv = d_nhwc(gfull, dt, 2 * Co, Co, seed + 1)
        a = _algo(lib, algo)

        def launch():
            dst = g_vec((Ci, Co, 2, 2), torch.float32)
            d = ops.make_gconv(ops._DT[dt], a, B, h, w_, Ci, ops.TAPS1, 1, (0, 0), h, w_, Ci, 4 * Co, 4, 2, off, H, W,
                               2 * Co)
            d.algo = a
            parts = _wgrad_call(lib, ops, bp, d, xv, gv, dst, 0, Co * 4, 1, 4, False)
            return [Out("dW", dst, ref, A, B * h * w_, "tf32" if _tf32(dt, algo) else "acc32"), Out("partials", parts)]
        return [xb, gb], launch
    return prepare


def outconv_fwd(dt, B, C, K, H, W, seed, ld=None):
    def prepare():
        lib, ops, UF, _ = _dev()
        g = _gen(seed)
        x = rq(torch.randn(B, C, H, W, generator=g), dt)
        w = torch.randn(K, C, generator=g) * 0.3
        b = torch.randn(K, generator=g)
        ref, A = ref_outconv(x, rq(w, dt), rq(b, dt))
        xb, xv = d_nhwc(x, dt, ld, 0, seed)
        wd, bd = w.to(DEV), b.to(DEV)

        def launch():
            lg = g_vec((B, H, W, K), dt)
            import ctypes as Cc
            lib.check(ops.lib().unetb200_outconv_fwd(ops._p(xv), ops.nhwc_ld(xv), ops._p(wd), ops._p(bd),
                                                     Cc.c_void_p(lg.ptr()), ops.dt(xv), B * H * W, C, K, ops._stream()),
                      "outconv_fwd")
            return [Out("logits", lg, ref.permute(0, 2, 3, 1), A.permute(0, 2, 3, 1), C + 1, _cname(dt))]
        return [xb, wd, bd], launch
    return prepare


def outconv_bwd(dt, B, C, K, H, W, seed, below=False, ld=None):
    """gx, dW, db of OutConv (and, with `below`, the BatchNorm + ReLU backward sums of the stage whose activation x
    is, from the same pass)"""
    def prepare():
        import ctypes as Cc
        lib, ops, UF, _ = _dev()
        g = _gen(seed)
        x = rq(torch.relu(torch.randn(B, C, H, W, generator=g)), dt)
        w = torch.randn(K, C, generator=g) * 0.3
        gl = rq(torch.randn(B, K, H, W, generator=g), dt)
        wq = rq(w, dt).double()
        gx_ref = torch.einsum("bkhw,kc->bchw", gl.double(), wq)
        gx_A = torch.einsum("bkhw,kc->bchw", gl.double().abs(), wq.abs())
        dw_ref = torch.einsum("bkhw,bchw->kc", gl.double(), x.double())
        dw_A = torch.einsum("bkhw,bchw->kc", gl.double().abs(), x.double().abs())
        db_ref, db_A = gl.double().sum((0, 2, 3)), gl.double().abs().sum((0, 2, 3))
        xb, xv = d_nhwc(x, dt, ld, 0, seed)
        glb = gl.permute(0, 2, 3, 1).contiguous().to(dt).to(DEV)
        wd = w.to(DEV)
        ins = [xb, glb, wd]
        if below:
            yprev = rq(torch.randn(B, C, H, W, generator=g), dt)
            coefs = _affine_coefs(g, C)
            yb, yv = d_nhwc(yprev, dt, seed=seed + 5)
            cd = coefs.to(DEV)
            ins += [yb, cd]
        L = ops.lib()

        def launch():
            gx = g_nhwc(B, C, H, W, dt)
            dw = g_vec((K, C), torch.float32)
            db = g_vec((K,), torch.float32)
            ws = torch.empty(L.unetb200_outconv_bwd_workspace(B * H * W, C, K), dtype=torch.float32, device=DEV)
            outs = [Out("gx", gx, gx_ref, gx_A, K, _cname(dt)),
                    Out("dW", dw, dw_ref, dw_A, B * H * W, "acc32", atomic=OUTCONV_ATOMIC),
                    Out("db", db, db_ref, db_A, B * H * W, "acc32", atomic=OUTCONV_ATOMIC)]
            if below:
                sums = g_vec((2, C), torch.float64, init=0.0)
                assert L.unetb200_outconv_bwd_bnbwd_supported(ops._p(xv), ops.nhwc_ld(xv), ops._p(gx.view), C, ops._p(yv),
                                                              ops.nhwc_ld(yv), ops.dt(xv), C, K), "fused OutConv backward not supported"
                lib.check(L.unetb200_outconv_bwd_bnbwd(ops._p(xv), ops.nhwc_ld(xv), ops._p(wd), ops._p(glb),
                                                       ops._p(gx.view), C, Cc.c_void_p(dw.ptr()), Cc.c_void_p(db.ptr()),
                                                       ops._p(ws), ops._p(yv), ops.nhwc_ld(yv), ops._p(cd),
                                                       Cc.c_void_p(sums.ptr()), ops.dt(xv), B * H * W, C, K, ops._stream()),
                          "outconv_bwd_bnbwd")
                torch.cuda.synchronize()
                sref, sA = ref_bnbwd_sums(gx.view.detach().double().cpu(), yprev, coefs)
                outs.append(Out("sums", sums, sref, sA, B * H * W, "acc32"))
            else:
                lib.check(L.unetb200_outconv_bwd(ops._p(xv), ops.nhwc_ld(xv), ops._p(wd), ops._p(glb), ops._p(gx.view), C,
                                                 Cc.c_void_p(dw.ptr()), Cc.c_void_p(db.ptr()), ops._p(ws), ops.dt(xv),
                                                 B * H * W, C, K, ops._stream()), "outconv_bwd")
            return outs
        return ins, launch
    return prepare


def pack_case(dt, kind, shape, seed, single=False, channels_last=False):
    """GEMM-operand packing of a weight (the operand every conv case reads): exact"""
    def prepare():
        lib, ops, UF, _ = _dev()
        g = _gen(seed)
        w = torch.randn(*shape, generator=g)
        wd = w.to(DEV)
        if channels_last:
            wd = wd.contiguous(memory_format=torch.channels_last)
        job = UF._JOBS[kind](wd)
        src, n, st, off, oshape = job
        if kind == "f3":
            ref = w.permute(0, 2, 3, 1).reshape(oshape)
        elif kind == "d3":
            ref = w.flip(2, 3).permute(1, 2, 3, 0).reshape(oshape)
        elif kind == "fT":
            ref = w.permute(2, 3, 1, 0).reshape(oshape)
        else:
            ref = w.permute(0, 2, 3, 1).reshape(oshape)
        ref = rq(ref, dt).double()

        def launch():
            import ctypes as C
            out = g_vec(oshape, dt)
            if single:
                lib.check(ops.lib().unetb200_pack_weights(ops._p(src), C.c_void_p(out.ptr()), ops._DT[dt], n[0], n[1], n[2],
                                                          st[0], st[1], st[2], off, ops._stream()), "pack_weights")
            else:
                jobs = (lib.PackJob * 1)()
                jobs[0].src, jobs[0].dst = src.data_ptr(), out.ptr()
                jobs[0].n0, jobs[0].n1, jobs[0].n2 = n
                jobs[0].s0, jobs[0].s1, jobs[0].s2 = st
                jobs[0].off = off
                lib.check(ops.lib().unetb200_pack_weights_multi(jobs, 1, ops._DT[dt], ops._stream()), "pack_weights_multi")
            return [Out("packed", out, ref, torch.zeros_like(ref), 1, "fp32")]
        return [wd], launch
    return prepare


# ------------------------------------------------------------------------------------------------
# the cases, by switch set
# ------------------------------------------------------------------------------------------------
# each set's switches are read once into statics by the library: the non-default sets run in a process of their own
ENV_SETS = {
    "default": {},
    "tc3_cg1": {"UNETB200_TC3_CG1": "1", "UNETB200_TC3_MAXBN": "256"},
    "tc3_maxbn256": {"UNETB200_TC3_MAXBN": "256"},
    "tc3w_stages5": {"UNETB200_TC3W_STAGES": "5"},
    "bnbwd64_cfg0": {"UNETB200_BNBWD64_CFG": "0"},
    "tc4w_all": {"UNETB200_TC4W": "all"},
    "no_halo": {"UNETB200_NO_HALO": "1", "UNETB200_NO_HALO_WGRAD": "1", "UNETB200_NO_FIRST_NARROW": "1",
                "UNETB200_NO_FIRST_TC": "1"},
}


def _shape(B, Ci, Co, H, W):
    return f"{B}x{Ci}>{Co}x{H}x{W}"


def _c3(out, env, dt, algo, B, Ci, Co, H, W, seed, ops=("f", "d", "w"), tag="", **kw):
    n = _cname(dt)
    s = _shape(B, Ci, Co, H, W) + tag
    if "f" in ops:
        out.append(Case(f"fprop:{n}:{algo}:{s}", conv3x3_fprop(dt, algo, B, Ci, Co, H, W, seed, **kw.get("f", {})), env))
    if "d" in ops:
        out.append(Case(f"dgrad:{n}:{algo}:{s}", conv3x3_dgrad(dt, algo, B, Ci, Co, H, W, seed + 1, **kw.get("d", {})), env))
    for lay in ("oihw", "cl", "multi"):
        if (lay == "oihw" and "w" in ops) or (lay != "oihw" and lay in ops):
            out.append(Case(f"wgrad_{lay}:{n}:{algo}:{s}",
                            conv3x3_wgrad(dt, algo, B, Ci, Co, H, W, seed + 2, layout=lay, **kw.get("w", {})), env))
    if "a" in ops:
        out.append(Case(f"affine:{n}:{algo}:{s}", conv3x3_affine(dt, algo, B, Ci, Co, H, W, seed + 3, **kw.get("a", {})), env))
    if "p" in ops:
        out.append(Case(f"affine_pool:{n}:{algo}:{s}", conv3x3_affine(dt, algo, B, Ci, Co, H, W, seed + 4, pool=True), env))
    if "b" in ops:
        out.append(Case(f"dgrad_bnbwd:{n}:{algo}:{s}", conv3x3_bnbwd(dt, algo, B, Ci, Co, H, W, seed + 5, **kw.get("b", {})), env))


def _ct(out, env, dt, algo, B, Ci, Co, h, w, seed, pad=(0, 0), ops="fdw"):
    n = _cname(dt)
    s = f"{B}x{Ci}>{Co}x{h}x{w}" + (f"_pad{pad[0]}{pad[1]}" if pad != (0, 0) else "")
    if "f" in ops:
        out.append(Case(f"convT_fprop:{n}:{algo}:{s}", convT_fprop(dt, algo, B, Ci, Co, h, w, seed, pad), env))
    if "d" in ops:
        out.append(Case(f"convT_dgrad:{n}:{algo}:{s}", convT_dgrad(dt, algo, B, Ci, Co, h, w, seed + 1, pad), env))
    if "w" in ops:
        out.append(Case(f"convT_wgrad:{n}:{algo}:{s}", convT_wgrad(dt, algo, B, Ci, Co, h, w, seed + 2, pad), env))


def build_cases():
    cs = []
    E = "default"
    sl = dict(f=dict(ld_in=96, c0_in=16, ld_out=160, c0_out=32), d=dict(ld_out=160, c0_out=64),
              w=dict(ld_in=96, c0_in=16))
    # ---- CTA-pair tcgen05 engine (conv_tc3.cu), bf16 and TF32: N blocks 64 / 128, ragged 16x16 tiles with an odd
    # tile count (a pair with one tile), W <= 8 (stacked sub-tiles), several tiles per CTA, slices in and out
    _c3(cs, E, BF, "tc", 1, 128, 64, 40, 36, 1000, ops=("f", "d", "w", "cl", "a", "p", "b"))
    _c3(cs, E, BF, "tc", 2, 128, 128, 20, 28, 1010, ops=("f", "d", "w", "multi", "a", "p", "b"))
    _c3(cs, E, BF, "tc", 3, 64, 128, 20, 8, 1020, ops=("f", "d", "a", "p", "b"))
    _c3(cs, E, BF, "tc", 2, 128, 128, 96, 96, 1030, ops=("f",))                          # 72 tiles: ring wrap
    _c3(cs, E, BF, "tc", 1, 64, 128, 17, 21, 1040, ops=("f", "d", "w"), tag="_slice", **sl)
    _c3(cs, E, BF, "tc", 1, 256, 256, 12, 10, 1050, ops=("f", "d", "w", "cl"))
    _c3(cs, E, BF, "tc", 3, 512, 256, 16, 8, 1060, ops=("w", "cl"))                      # CTA-pair wgrad, odd batch
    _c3(cs, E, FP, "tc", 1, 64, 64, 19, 21, 1070, ops=("f", "d", "w", "a", "b"))
    _c3(cs, E, FP, "tc", 2, 128, 128, 10, 12, 1080, ops=("f", "d", "w", "cl", "a", "b"))
    _c3(cs, E, FP, "tc", 1, 128, 64, 7, 9, 1090, ops=("f", "d"), tag="_slice",
        f=dict(ld_in=160, c0_in=16, ld_out=96, c0_out=32), d=dict(ld_out=160, c0_out=16))
    _c3(cs, E, BF, "tc", 2, 64, 128, 12, 20, 1095, ops=("f",), tag="_bias", f=dict(bias=True))     # bias: tc2 + stats
    for i, ncls in enumerate(range(1, 9)):                                               # fused inference head
        cs.append(Case(f"head:bf16:tc:{_shape(1 + i % 2, 64 * (1 + i % 2), 64, 17 + i, 20)}:k{ncls}",
                       conv3x3_head(1 + i % 2, 64 * (1 + i % 2), 17 + i, 20, ncls, 1100 + i, bias=(ncls != 3))))
    # ---- persistent engine (conv_tc2.cu): ConvTranspose (4 quadrants), its 4-tap dgrad, its wgrad; bias
    for i, (B, Ci, Co, h, w, pad) in enumerate([(2, 64, 64, 7, 9, (0, 0)), (1, 256, 128, 5, 4, (1, 1)),
                                                (1, 512, 256, 4, 4, (0, 0)), (2, 128, 128, 9, 7, (1, 0))]):
        _ct(cs, E, BF, "tc", B, Ci, Co, h, w, 1200 + 10 * i, pad)
    _ct(cs, E, BF, "tc", 2, 128, 64, 6, 10, 1250)
    for i, (B, Ci, Co, h, w, pad) in enumerate([(2, 64, 64, 6, 5, (0, 0)), (1, 128, 64, 4, 4, (1, 0)),
                                                (1, 256, 128, 5, 6, (0, 1))]):
        _ct(cs, E, FP, "tc", B, Ci, Co, h, w, 1300 + 10 * i, pad)
    # ---- N-stacked wgrad (conv_tc4.cu) and the remaining tcgen05 wgrads
    _c3(cs, E, BF, "tc", 2, 128, 64, 24, 20, 1400, ops=("w", "cl"))
    _c3(cs, E, BF, "tc", 1, 64, 64, 33, 17, 1410, ops=("w",))
    _c3(cs, E, FP, "tc", 2, 64, 128, 12, 12, 1420, ops=("w",))
    _c3(cs, E, BF, "tc", 2, 64, 64, 64, 64, 1430, ops=("w", "cl"))          # channels_last, 8 <= splits < 32
    _c3(cs, E, BF, "tc", 2, 128, 128, 32, 48, 1440, ops=("w", "cl"))
    _c3(cs, E, BF, "tc", 2, 64, 64, 128, 128, 1450, ops=("cl",))            # channels_last, >= 32 splits
    # ---- TMA-staged narrow engine (conv_halo.cu): every channel pair, plain / affine / BatchNorm-backward
    # epilogues, TF32 (ES = 4), 8-channel tensors on the 16-channel instantiations, several tiles per CTA
    for i, (Ci, Co) in enumerate([(16, 16), (16, 32), (16, 64), (32, 16), (32, 32), (32, 64), (64, 16), (64, 32)]):
        B, H, W = (1, 33, 20) if i % 2 else (2, 24, 17)
        _c3(cs, E, BF, "auto", B, Ci, Co, H, W, 1500 + 10 * i, ops=("f", "w", "a"))
    for i, (Ci, Co) in enumerate([(16, 16), (16, 32), (32, 16), (32, 32), (64, 16), (64, 32)]):
        _c3(cs, E, BF, "auto", 2, Co, Ci, 18, 22, 1600 + 10 * i, ops=("b",))            # dgrad N = Ci
    _c3(cs, E, BF, "auto", 8, 16, 16, 128, 128, 1700, ops=("f", "d", "w"))               # many tiles per CTA
    _c3(cs, E, BF, "auto", 2, 8, 8, 37, 41, 1710, ops=("f", "d", "w", "a", "b"))
    _c3(cs, E, BF, "auto", 1, 16, 8, 20, 24, 1720, ops=("f", "w"))
    _c3(cs, E, BF, "auto", 2, 32, 32, 16, 16, 1730, ops=("f", "w"), tag="_slice",
        f=dict(ld_in=64, c0_in=16, ld_out=96, c0_out=64), w=dict(ld_in=64, c0_in=16))
    _c3(cs, E, BF, "auto", 2, 16, 32, 16, 24, 1740, ops=("p",))
    for i, (Ci, Co) in enumerate([(16, 16), (16, 32), (32, 16), (32, 32)]):
        _c3(cs, E, FP, "prefer", 1, Ci, Co, 21, 19, 1800 + 10 * i, ops=("f", "d", "a"))
    # ---- narrow ConvTranspose (conv_halo_t.cu)
    for i, (Ci, Co) in enumerate([(16, 8), (32, 16), (32, 32), (64, 16), (64, 32)]):
        _ct(cs, E, BF, "tc", 1 + i % 2, Ci, Co, 9 + i, 7 + i, 1900 + 10 * i)
    _ct(cs, E, BF, "auto", 2, 32, 16, 5, 6, 1990, pad=(1, 2), ops="f")
    # ---- first layers: C_in = 1..4 -> 64 on the tensor cores (conv_first_tc.cu), C_in = 1 -> 8 / 16 / 32 on the
    # CUDA cores (conv_first_narrow.cu), and the exact CUDA-core kernels (conv_first.cu)
    for cin in (1, 2, 3, 4):
        _c3(cs, E, BF, "auto", 2, cin, 64, 30, 34, 2000 + 10 * cin, ops=("f", "a", "w"))
    for co in (8, 16, 32):
        _c3(cs, E, BF, "auto", 2, 1, co, 37, 45, 2100 + co, ops=("f", "a", "w"))
    for dt in (FP, BF):
        _c3(cs, E, dt, "simt", 2, 1, 64, 20, 22, 2200, ops=("f", "w"))                    # tiled
        _c3(cs, E, dt, "simt", 1, 1, 128, 9, 13, 2210, ops=("f", "w"))
        for cin in (2, 3, 4):
            _c3(cs, E, dt, "simt", 1, cin, 32, 12, 16, 2220 + cin, ops=("f", "w"))      # px4 (W % 4 == 0)
            _c3(cs, E, dt, "simt", 1, cin, 32, 11, 13, 2230 + cin, ops=("f",))           # W % 4 != 0
    # ---- CUDA-core implicit GEMM (conv_simt.cu): vector / scalar loads, N blocks 16 / 32 / 64
    for dt in (FP, BF):
        for i, (Ci, Co) in enumerate([(48, 12), (48, 24), (48, 80), (6, 12), (6, 24), (6, 80)]):
            _c3(cs, E, dt, "simt", 2, Ci, Co, 9, 11, 2300 + 10 * i + (dt == BF), ops=("f", "w"))
        _c3(cs, E, dt, "simt", 1, 64, 64, 8, 8, 2400 + (dt == BF), ops=("f", "d", "w"), tag="_slice", **sl)
        _ct(cs, E, dt, "simt", 2, 32, 16, 4, 5, 2410 + (dt == BF), pad=(1, 2))
    # ---- exact-fp32 narrow kernels (conv_simt_narrow.cu)
    for i, (Ci, Co) in enumerate([(16, 16), (16, 32), (16, 64), (32, 16), (32, 32), (32, 64), (64, 16), (64, 32)]):
        _c3(cs, E, FP, "simt", 1, Ci, Co, 17, 23, 2500 + 10 * i, ops=("f", "w"))
    for i, (Ci, Co) in enumerate([(64, 8), (32, 8), (16, 8), (8, 64), (8, 32), (8, 16), (8, 8)]):
        _c3(cs, E, FP, "simt", 2, Ci, Co, 13, 19, 2600 + 10 * i, ops=("w",))
    # ---- OutConv (outconv.cu): n_classes 1..8 and more, C % 8 != 0 (scalar), slice input, fused BatchNorm backward
    for dt in (FP, BF):
        for K in range(1, 9):
            C = 64 if K % 2 else 16
            cs.append(Case(f"outconv_fwd:{_cname(dt)}:{1 + K % 2}x{C}>{K}x{9 + K}x{7 + K}",
                           outconv_fwd(dt, 1 + K % 2, C, K, 9 + K, 7 + K, 2700 + K, ld=(C + 16) if K == 5 else None)))
            for below in (False, True):
                cs.append(Case(f"outconv_bwd{'_bnbwd' if below else ''}:{_cname(dt)}:{1 + K % 2}x{C}>{K}x{10 + K}x{7 + K}",
                               outconv_bwd(dt, 1 + K % 2, C, K, 10 + K, 7 + K, 2800 + 2 * K + below, below=below)))
        cs.append(Case(f"outconv_fwd:{_cname(dt)}:1x6>3x7x9", outconv_fwd(dt, 1, 6, 3, 7, 9, 2900)))
        cs.append(Case(f"outconv_bwd:{_cname(dt)}:1x6>3x7x9", outconv_bwd(dt, 1, 6, 3, 7, 9, 2901)))
    # ---- weight packing
    for dt in (FP, BF):
        n = _cname(dt)
        cs.append(Case(f"pack_multi:{n}:f3", pack_case(dt, "f3", (32, 16, 3, 3), 3000)))
        cs.append(Case(f"pack_single:{n}:d3", pack_case(dt, "d3", (24, 40, 3, 3), 3001, single=True)))
        cs.append(Case(f"pack_single:{n}:d3_cl", pack_case(dt, "d3", (64, 48, 3, 3), 3002, single=True, channels_last=True)))

    # ---- switch sets
    E = "tc3_cg1"
    _c3(cs, E, BF, "tc", 1, 128, 64, 40, 36, 4000, ops=("f", "a"))
    _c3(cs, E, BF, "tc", 3, 64, 128, 20, 8, 4010, ops=("f", "a"))
    _c3(cs, E, BF, "tc", 1, 256, 256, 12, 10, 4020, ops=("f",))
    _c3(cs, E, FP, "tc", 1, 128, 64, 19, 21, 4030, ops=("f", "a"))
    _c3(cs, E, FP, "tc", 2, 128, 128, 10, 12, 4040, ops=("f", "a"))
    E = "tc3_maxbn256"
    _c3(cs, E, BF, "tc", 1, 256, 256, 12, 10, 4100, ops=("f",))
    _c3(cs, E, BF, "tc", 2, 128, 256, 17, 9, 4110, ops=("f",))
    E = "tc3w_stages5"
    _c3(cs, E, BF, "tc", 1, 256, 256, 12, 10, 4200, ops=("w",))
    E = "bnbwd64_cfg0"
    _c3(cs, E, BF, "tc", 1, 64, 128, 40, 36, 4300, ops=("b",))              # dgrad 128 -> 64: N block 64
    E = "tc4w_all"
    _c3(cs, E, BF, "tc", 1, 256, 256, 12, 10, 4400, ops=("w",))
    E = "no_halo"
    _c3(cs, E, BF, "simt", 2, 1, 64, 20, 22, 4990, ops=("f",))               # bf16 tiled first layer
    for i, cin in enumerate((1, 2, 3, 4, 8, 16, 32, 64)):
        for j, co in enumerate((16, 32, 64)):
            if (cin == 64 and co == 64) or (cin <= 4 and co == 64):     # the pair kernel's / conv_first_tc.cu's
                continue
            sd = 5000 + 10 * (3 * i + j)
            _c3(cs, E, BF, "auto", 1, cin, co, 13 + j, 11 + i, sd, ops=("f", "a", "w"))
    return cs


CASES = build_cases()


# ------------------------------------------------------------------------------------------------
# the ledger: normalised kernel name -> the cases that launch it (a tuple of case ids), ("env", switches, cases) for
# a kernel only some switch set reaches, or ("unreachable", reason) for one no route reaches under any switch
# ------------------------------------------------------------------------------------------------
LEDGER = {
    'tc2_wgrad_kernel<float, 64, 3>': (
        'convT_wgrad:fp32:tc:1x128>64x4x4_pad10',
        'convT_wgrad:fp32:tc:2x64>64x6x5',
        'wgrad_oihw:fp32:tc:1x64>64x19x21',
    ),
    'tc2_wgrad_kernel<float, 128, 3>': (
        'convT_wgrad:fp32:tc:1x256>128x5x6_pad01',
        'wgrad_cl:fp32:tc:2x128>128x10x12',
        'wgrad_oihw:fp32:tc:2x128>128x10x12',
        'wgrad_oihw:fp32:tc:2x64>128x12x12',
    ),
    'tc2_wgrad_kernel<__nv_bfloat16, 64, 6>': (
        'convT_wgrad:bf16:tc:2x128>64x6x10',
        'convT_wgrad:bf16:tc:2x64>64x7x9',
    ),
    'tc2_wgrad_kernel<__nv_bfloat16, 128, 5>': (
        'convT_wgrad:bf16:tc:1x256>128x5x4_pad11',
        'convT_wgrad:bf16:tc:1x512>256x4x4',
        'convT_wgrad:bf16:tc:2x128>128x9x7_pad10',
    ),
    'tc2_fprop_kernel<float, 64, 3, 6, 2>': (
        'convT_dgrad:fp32:tc:2x64>64x6x5',
    ),
    'tc2_fprop_kernel<float, 128, 3, 4, 2>': (
        'convT_dgrad:fp32:tc:1x128>64x4x4_pad10',
        'convT_dgrad:fp32:tc:1x256>128x5x6_pad01',
        'convT_fprop:fp32:tc:1x128>64x4x4_pad10',
        'convT_fprop:fp32:tc:1x256>128x5x6_pad01',
        'convT_fprop:fp32:tc:2x64>64x6x5',
    ),
    'tc2_fprop_kernel<__nv_bfloat16, 64, 3, 6, 2>': (
        'convT_dgrad:bf16:tc:2x64>64x7x9',
    ),
    'tc2_fprop_kernel<__nv_bfloat16, 128, 3, 4, 2>': (
        'convT_dgrad:bf16:tc:2x128>128x9x7_pad10',
        'convT_dgrad:bf16:tc:2x128>64x6x10',
        'convT_fprop:bf16:tc:1x256>128x5x4_pad11',
        'convT_fprop:bf16:tc:1x512>256x4x4',
        'convT_fprop:bf16:tc:2x128>128x9x7_pad10',
        'convT_fprop:bf16:tc:2x128>64x6x10',
        'convT_fprop:bf16:tc:2x64>64x7x9',
        'fprop:bf16:tc:2x64>128x12x20_bias',
    ),
    'tc2_fprop_kernel<__nv_bfloat16, 256, 2, 3, 1>': (
        'convT_dgrad:bf16:tc:1x256>128x5x4_pad11',
        'convT_dgrad:bf16:tc:1x512>256x4x4',
    ),
    'tc2_stats_reduce_kernel': (
        'fprop:bf16:tc:2x64>128x12x20_bias',
    ),
    'tc3_conv_kernel<float, 64, 3, 6, 2, 1, 1, 0>': ("env", {'UNETB200_TC3_CG1': '1', 'UNETB200_TC3_MAXBN': '256'}, (
        'tc3_cg1/fprop:fp32:tc:1x128>64x19x21',
    )),
    'tc3_conv_kernel<float, 128, 2, 6, 2, 1, 1, 0>': ("env", {'UNETB200_TC3_CG1': '1', 'UNETB200_TC3_MAXBN': '256'}, (
        'tc3_cg1/fprop:fp32:tc:2x128>128x10x12',
    )),
    'tc3_conv_kernel<float, 64, 3, 3, 2, 2, 3, 0>': (
        'dgrad:fp32:tc:1x64>64x19x21',
        'fprop:fp32:tc:1x128>64x7x9_slice',
        'fprop:fp32:tc:1x64>64x19x21',
    ),
    'tc3_conv_kernel<float, 128, 2, 3, 2, 2, 3, 0>': (
        'dgrad:fp32:tc:1x128>64x7x9_slice',
        'dgrad:fp32:tc:2x128>128x10x12',
        'fprop:fp32:tc:2x128>128x10x12',
    ),
    'tc3_conv_kernel<__nv_bfloat16, 64, 3, 6, 2, 1, 1, 0>': ("env", {'UNETB200_TC3_CG1': '1', 'UNETB200_TC3_MAXBN': '256'}, (
        'tc3_cg1/fprop:bf16:tc:1x128>64x40x36',
    )),
    'tc3_conv_kernel<__nv_bfloat16, 128, 2, 6, 2, 1, 1, 0>': ("env", {'UNETB200_TC3_CG1': '1', 'UNETB200_TC3_MAXBN': '256'}, (
        'tc3_cg1/fprop:bf16:tc:3x64>128x20x8',
    )),
    'tc3_conv_kernel<__nv_bfloat16, 256, 2, 3, 1, 1, 1, 0>': ("env", {'UNETB200_TC3_CG1': '1', 'UNETB200_TC3_MAXBN': '256'}, (
        'tc3_cg1/fprop:bf16:tc:1x256>256x12x10',
    )),
    'tc3_conv_kernel<__nv_bfloat16, 64, 3, 3, 2, 2, 3, 0>': (
        'dgrad:bf16:tc:1x64>128x17x21_slice',
        'dgrad:bf16:tc:3x64>128x20x8',
        'fprop:bf16:tc:1x128>64x40x36',
    ),
    'tc3_conv_kernel<__nv_bfloat16, 128, 2, 3, 2, 2, 3, 0>': (
        'dgrad:bf16:tc:1x128>64x40x36',
        'dgrad:bf16:tc:1x256>256x12x10',
        'dgrad:bf16:tc:2x128>128x20x28',
        'fprop:bf16:tc:1x256>256x12x10',
        'fprop:bf16:tc:1x64>128x17x21_slice',
        'fprop:bf16:tc:2x128>128x20x28',
        'fprop:bf16:tc:2x128>128x96x96',
        'fprop:bf16:tc:3x64>128x20x8',
    ),
    'tc3_conv_kernel<__nv_bfloat16, 256, 2, 2, 1, 2, 3, 0>': ("env", {'UNETB200_TC3_MAXBN': '256'}, (
        'tc3_maxbn256/fprop:bf16:tc:1x256>256x12x10',
        'tc3_maxbn256/fprop:bf16:tc:2x128>256x17x9',
    )),
    'tc3_conv_kernel<float, 64, 3, 2, 2, 2, 3, 2>': (
        'dgrad_bnbwd:fp32:tc:1x64>64x19x21',
    ),
    'tc3_conv_kernel<float, 128, 2, 3, 2, 2, 3, 2>': (
        'dgrad_bnbwd:fp32:tc:2x128>128x10x12',
    ),
    'tc3_conv_kernel<__nv_bfloat16, 64, 2, 3, 2, 2, 3, 2>': ("env", {'UNETB200_BNBWD64_CFG': '0'}, (
        'bnbwd64_cfg0/dgrad_bnbwd:bf16:tc:1x64>128x40x36',
    )),
    'tc3_conv_kernel<__nv_bfloat16, 64, 3, 2, 2, 2, 3, 2>': (
        'dgrad_bnbwd:bf16:tc:3x64>128x20x8',
    ),
    'tc3_conv_kernel<__nv_bfloat16, 128, 2, 3, 2, 2, 3, 2>': (
        'dgrad_bnbwd:bf16:tc:1x128>64x40x36',
        'dgrad_bnbwd:bf16:tc:2x128>128x20x28',
    ),
    'tc3_conv_kernel<float, 64, 3, 6, 2, 1, 1, 1>': ("env", {'UNETB200_TC3_CG1': '1', 'UNETB200_TC3_MAXBN': '256'}, (
        'tc3_cg1/affine:fp32:tc:1x128>64x19x21',
    )),
    'tc3_conv_kernel<float, 128, 2, 6, 2, 1, 1, 1>': ("env", {'UNETB200_TC3_CG1': '1', 'UNETB200_TC3_MAXBN': '256'}, (
        'tc3_cg1/affine:fp32:tc:2x128>128x10x12',
    )),
    'tc3_conv_kernel<float, 64, 3, 3, 2, 2, 3, 1>': (
        'affine:fp32:tc:1x64>64x19x21',
    ),
    'tc3_conv_kernel<float, 128, 2, 3, 2, 2, 3, 1>': (
        'affine:fp32:tc:2x128>128x10x12',
    ),
    'tc3_conv_kernel<__nv_bfloat16, 64, 3, 6, 2, 1, 1, 1>': ("env", {'UNETB200_TC3_CG1': '1', 'UNETB200_TC3_MAXBN': '256'}, (
        'tc3_cg1/affine:bf16:tc:1x128>64x40x36',
    )),
    'tc3_conv_kernel<__nv_bfloat16, 128, 2, 6, 2, 1, 1, 1>': ("env", {'UNETB200_TC3_CG1': '1', 'UNETB200_TC3_MAXBN': '256'}, (
        'tc3_cg1/affine:bf16:tc:3x64>128x20x8',
    )),
    'tc3_conv_kernel<__nv_bfloat16, 64, 3, 3, 2, 2, 3, 1>': (
        'affine:bf16:tc:1x128>64x40x36',
        'affine_pool:bf16:tc:1x128>64x40x36',
    ),
    'tc3_conv_kernel<__nv_bfloat16, 128, 2, 3, 2, 2, 3, 1>': (
        'affine:bf16:tc:2x128>128x20x28',
        'affine:bf16:tc:3x64>128x20x8',
        'affine_pool:bf16:tc:2x128>128x20x28',
        'affine_pool:bf16:tc:3x64>128x20x8',
    ),
    'tc3_conv_kernel<__nv_bfloat16, 64, 3, 3, 2, 2, 3, 3>': (
        'head:bf16:tc:1x64>64x17x20:k1',
        'head:bf16:tc:1x64>64x19x20:k3',
        'head:bf16:tc:1x64>64x21x20:k5',
        'head:bf16:tc:1x64>64x23x20:k7',
        'head:bf16:tc:2x128>64x18x20:k2',
        'head:bf16:tc:2x128>64x20x20:k4',
        'head:bf16:tc:2x128>64x22x20:k6',
        'head:bf16:tc:2x128>64x24x20:k8',
    ),
    'tc3_wgrad_kernel<5>': ("env", {'UNETB200_TC3W_STAGES': '5'}, (
        'tc3w_stages5/wgrad_oihw:bf16:tc:1x256>256x12x10',
    )),
    'tc3_wgrad_kernel<7>': (
        'wgrad_cl:bf16:tc:1x256>256x12x10',
        'wgrad_cl:bf16:tc:3x512>256x16x8',
        'wgrad_oihw:bf16:tc:1x256>256x12x10',
        'wgrad_oihw:bf16:tc:3x512>256x16x8',
    ),
    'tc3_stats_reduce_kernel': (
        'dgrad_bnbwd:bf16:tc:1x128>64x40x36',
        'dgrad_bnbwd:bf16:tc:2x128>128x20x28',
        'dgrad_bnbwd:bf16:tc:3x64>128x20x8',
        'dgrad_bnbwd:fp32:tc:1x64>64x19x21',
        'dgrad_bnbwd:fp32:tc:2x128>128x10x12',
        'fprop:bf16:tc:1x128>64x40x36',
        'fprop:bf16:tc:1x256>256x12x10',
        'fprop:bf16:tc:1x64>128x17x21_slice',
        'fprop:bf16:tc:2x128>128x20x28',
        'fprop:bf16:tc:2x128>128x96x96',
        'fprop:bf16:tc:3x64>128x20x8',
        'fprop:fp32:tc:1x128>64x7x9_slice',
        'fprop:fp32:tc:1x64>64x19x21',
        'fprop:fp32:tc:2x128>128x10x12',
        'bnbwd64_cfg0/dgrad_bnbwd:bf16:tc:1x64>128x40x36',
        'tc3_cg1/fprop:bf16:tc:1x128>64x40x36',
        'tc3_cg1/fprop:bf16:tc:1x256>256x12x10',
        'tc3_cg1/fprop:bf16:tc:3x64>128x20x8',
        'tc3_cg1/fprop:fp32:tc:1x128>64x19x21',
        'tc3_cg1/fprop:fp32:tc:2x128>128x10x12',
        'tc3_maxbn256/fprop:bf16:tc:1x256>256x12x10',
        'tc3_maxbn256/fprop:bf16:tc:2x128>256x17x9',
    ),
    'tc4_wgrad_kernel<10>': (
        'wgrad_cl:bf16:tc:1x128>64x40x36',
        'wgrad_cl:bf16:tc:2x128>128x32x48',
        'wgrad_cl:bf16:tc:2x128>64x24x20',
        'wgrad_cl:bf16:tc:2x64>64x128x128',
        'wgrad_cl:bf16:tc:2x64>64x64x64',
        'wgrad_multi:bf16:tc:2x128>128x20x28',
        'wgrad_oihw:bf16:tc:1x128>64x40x36',
        'wgrad_oihw:bf16:tc:1x64>128x17x21_slice',
        'wgrad_oihw:bf16:tc:1x64>64x33x17',
        'wgrad_oihw:bf16:tc:2x128>128x20x28',
        'wgrad_oihw:bf16:tc:2x128>128x32x48',
        'wgrad_oihw:bf16:tc:2x128>64x24x20',
        'wgrad_oihw:bf16:tc:2x64>64x64x64',
        'tc4w_all/wgrad_oihw:bf16:tc:1x256>256x12x10',
    ),
    'halo_wgrad_kernel<64, 32>': (
        'wgrad_oihw:bf16:auto:1x64>32x33x20',
    ),
    'halo_wgrad_kernel<64, 16>': (
        'wgrad_oihw:bf16:auto:2x64>16x24x17',
    ),
    'halo_wgrad_kernel<32, 64>': (
        'wgrad_oihw:bf16:auto:1x32>64x33x20',
    ),
    'halo_wgrad_kernel<32, 32>': (
        'wgrad_oihw:bf16:auto:2x32>32x16x16_slice',
        'wgrad_oihw:bf16:auto:2x32>32x24x17',
    ),
    'halo_wgrad_kernel<32, 16>': (
        'wgrad_oihw:bf16:auto:1x32>16x33x20',
    ),
    'halo_wgrad_kernel<16, 64>': (
        'wgrad_oihw:bf16:auto:2x16>64x24x17',
    ),
    'halo_wgrad_kernel<16, 32>': (
        'wgrad_oihw:bf16:auto:1x16>32x33x20',
    ),
    'halo_wgrad_kernel<16, 16>': (
        'wgrad_oihw:bf16:auto:1x16>8x20x24',
        'wgrad_oihw:bf16:auto:2x16>16x24x17',
        'wgrad_oihw:bf16:auto:2x8>8x37x41',
        'wgrad_oihw:bf16:auto:8x16>16x128x128',
    ),
    'halo_conv_kernel<64, 32, 0, 2>': (
        'fprop:bf16:auto:1x64>32x33x20',
    ),
    'halo_conv_kernel<64, 16, 0, 2>': (
        'fprop:bf16:auto:2x64>16x24x17',
    ),
    'halo_conv_kernel<64, 32, 1, 2>': (
        'affine:bf16:auto:1x64>32x33x20',
    ),
    'halo_conv_kernel<64, 16, 1, 2>': (
        'affine:bf16:auto:2x64>16x24x17',
    ),
    'halo_conv_kernel<32, 64, 0, 2>': (
        'fprop:bf16:auto:1x32>64x33x20',
    ),
    'halo_conv_kernel<32, 32, 0, 2>': (
        'fprop:bf16:auto:2x32>32x16x16_slice',
        'fprop:bf16:auto:2x32>32x24x17',
    ),
    'halo_conv_kernel<32, 16, 0, 2>': (
        'fprop:bf16:auto:1x32>16x33x20',
    ),
    'halo_conv_kernel<32, 64, 1, 2>': (
        'affine:bf16:auto:1x32>64x33x20',
    ),
    'halo_conv_kernel<32, 32, 1, 2>': (
        'affine:bf16:auto:2x32>32x24x17',
    ),
    'halo_conv_kernel<32, 16, 1, 2>': (
        'affine:bf16:auto:1x32>16x33x20',
    ),
    'halo_conv_kernel<16, 64, 0, 2>': (
        'fprop:bf16:auto:2x16>64x24x17',
    ),
    'halo_conv_kernel<16, 32, 0, 2>': (
        'fprop:bf16:auto:1x16>32x33x20',
    ),
    'halo_conv_kernel<16, 16, 0, 2>': (
        'dgrad:bf16:auto:2x8>8x37x41',
        'dgrad:bf16:auto:8x16>16x128x128',
        'fprop:bf16:auto:1x16>8x20x24',
        'fprop:bf16:auto:2x16>16x24x17',
        'fprop:bf16:auto:2x8>8x37x41',
        'fprop:bf16:auto:8x16>16x128x128',
    ),
    'halo_conv_kernel<16, 64, 1, 2>': (
        'affine:bf16:auto:2x16>64x24x17',
    ),
    'halo_conv_kernel<16, 32, 1, 2>': (
        'affine:bf16:auto:1x16>32x33x20',
        'affine_pool:bf16:auto:2x16>32x16x24',
    ),
    'halo_conv_kernel<16, 16, 1, 2>': (
        'affine:bf16:auto:2x16>16x24x17',
        'affine:bf16:auto:2x8>8x37x41',
    ),
    'halo_conv_kernel<32, 32, 0, 4>': (
        'dgrad:fp32:prefer:1x32>32x21x19',
        'fprop:fp32:prefer:1x32>32x21x19',
    ),
    'halo_conv_kernel<32, 16, 0, 4>': (
        'dgrad:fp32:prefer:1x16>32x21x19',
        'fprop:fp32:prefer:1x32>16x21x19',
    ),
    'halo_conv_kernel<32, 32, 1, 4>': (
        'affine:fp32:prefer:1x32>32x21x19',
    ),
    'halo_conv_kernel<32, 16, 1, 4>': (
        'affine:fp32:prefer:1x32>16x21x19',
    ),
    'halo_conv_kernel<16, 32, 0, 4>': (
        'dgrad:fp32:prefer:1x32>16x21x19',
        'fprop:fp32:prefer:1x16>32x21x19',
    ),
    'halo_conv_kernel<16, 16, 0, 4>': (
        'dgrad:fp32:prefer:1x16>16x21x19',
        'fprop:fp32:prefer:1x16>16x21x19',
    ),
    'halo_conv_kernel<16, 32, 1, 4>': (
        'affine:fp32:prefer:1x16>32x21x19',
    ),
    'halo_conv_kernel<16, 16, 1, 4>': (
        'affine:fp32:prefer:1x16>16x21x19',
    ),
    'halo_conv_kernel<64, 32, 2, 2>': (
        'dgrad_bnbwd:bf16:auto:2x32>64x18x22',
    ),
    'halo_conv_kernel<64, 16, 2, 2>': (
        'dgrad_bnbwd:bf16:auto:2x16>64x18x22',
    ),
    'halo_conv_kernel<32, 32, 2, 2>': (
        'dgrad_bnbwd:bf16:auto:2x32>32x18x22',
    ),
    'halo_conv_kernel<32, 16, 2, 2>': (
        'dgrad_bnbwd:bf16:auto:2x16>32x18x22',
    ),
    'halo_conv_kernel<16, 32, 2, 2>': (
        'dgrad_bnbwd:bf16:auto:2x32>16x18x22',
    ),
    'halo_conv_kernel<16, 16, 2, 2>': (
        'dgrad_bnbwd:bf16:auto:2x16>16x18x22',
        'dgrad_bnbwd:bf16:auto:2x8>8x37x41',
    ),
    'halo_t_wgrad_kernel<64, 32>': (
        'convT_wgrad:bf16:tc:1x64>32x13x11',
    ),
    'halo_t_wgrad_kernel<64, 16>': (
        'convT_wgrad:bf16:tc:2x64>16x12x10',
    ),
    'halo_t_wgrad_kernel<32, 32>': (
        'convT_wgrad:bf16:tc:1x32>32x11x9',
    ),
    'halo_t_wgrad_kernel<32, 16>': (
        'convT_wgrad:bf16:tc:2x32>16x10x8',
    ),
    'halo_t_wgrad_kernel<16, 16>': (
        'convT_wgrad:bf16:tc:1x16>8x9x7',
    ),
    'halo_t_dgrad_kernel<32, 64>': (
        'convT_dgrad:bf16:tc:1x64>32x13x11',
    ),
    'halo_t_dgrad_kernel<16, 64>': (
        'convT_dgrad:bf16:tc:2x64>16x12x10',
    ),
    'halo_t_dgrad_kernel<32, 32>': (
        'convT_dgrad:bf16:tc:1x32>32x11x9',
    ),
    'halo_t_dgrad_kernel<16, 32>': (
        'convT_dgrad:bf16:tc:1x16>8x9x7',
        'convT_dgrad:bf16:tc:2x32>16x10x8',
    ),
    'halo_t_fprop_kernel<64, 32>': (
        'convT_fprop:bf16:tc:1x64>32x13x11',
    ),
    'halo_t_fprop_kernel<64, 16>': (
        'convT_fprop:bf16:tc:2x64>16x12x10',
    ),
    'halo_t_fprop_kernel<32, 32>': (
        'convT_fprop:bf16:tc:1x32>32x11x9',
    ),
    'halo_t_fprop_kernel<32, 16>': (
        'convT_fprop:bf16:auto:2x32>16x5x6_pad12',
        'convT_fprop:bf16:tc:2x32>16x10x8',
    ),
    'halo_t_fprop_kernel<16, 16>': (
        'convT_fprop:bf16:tc:1x16>8x9x7',
    ),
    'first_tc_kernel<4, 0>': (
        'fprop:bf16:auto:2x4>64x30x34',
    ),
    'first_tc_kernel<4, 1>': (
        'affine:bf16:auto:2x4>64x30x34',
    ),
    'first_tc_kernel<3, 0>': (
        'fprop:bf16:auto:2x3>64x30x34',
    ),
    'first_tc_kernel<3, 1>': (
        'affine:bf16:auto:2x3>64x30x34',
    ),
    'first_tc_kernel<2, 0>': (
        'fprop:bf16:auto:2x2>64x30x34',
    ),
    'first_tc_kernel<2, 1>': (
        'affine:bf16:auto:2x2>64x30x34',
    ),
    'first_tc_kernel<1, 0>': (
        'fprop:bf16:auto:2x1>64x30x34',
        'fprop:bf16:simt:2x1>64x20x22',
    ),
    'first_tc_kernel<1, 1>': (
        'affine:bf16:auto:2x1>64x30x34',
    ),
    'first_narrow_wgrad_kernel<4>': (
        'wgrad_oihw:bf16:auto:2x1>32x37x45',
    ),
    'first_narrow_wgrad_kernel<2>': (
        'wgrad_oihw:bf16:auto:2x1>16x37x45',
    ),
    'first_narrow_wgrad_kernel<1>': (
        'wgrad_oihw:bf16:auto:2x1>8x37x45',
    ),
    'first_narrow_fprop_kernel<4, 0>': (
        'fprop:bf16:auto:2x1>32x37x45',
    ),
    'first_narrow_fprop_kernel<2, 0>': (
        'fprop:bf16:auto:2x1>16x37x45',
    ),
    'first_narrow_fprop_kernel<1, 0>': (
        'fprop:bf16:auto:2x1>8x37x45',
    ),
    'first_narrow_fprop_kernel<4, 1>': (
        'affine:bf16:auto:2x1>32x37x45',
    ),
    'first_narrow_fprop_kernel<2, 1>': (
        'affine:bf16:auto:2x1>16x37x45',
    ),
    'first_narrow_fprop_kernel<1, 1>': (
        'affine:bf16:auto:2x1>8x37x45',
    ),
    'narrow_wgrad_kernel<64, 32>': ("env", {'UNETB200_NO_HALO': '1', 'UNETB200_NO_HALO_WGRAD': '1', 'UNETB200_NO_FIRST_NARROW': '1', 'UNETB200_NO_FIRST_TC': '1'}, (
        'no_halo/wgrad_oihw:bf16:auto:1x64>32x14x18',
    )),
    'narrow_wgrad_kernel<64, 16>': ("env", {'UNETB200_NO_HALO': '1', 'UNETB200_NO_HALO_WGRAD': '1', 'UNETB200_NO_FIRST_NARROW': '1', 'UNETB200_NO_FIRST_TC': '1'}, (
        'no_halo/wgrad_oihw:bf16:auto:1x64>16x13x18',
    )),
    'narrow_wgrad_kernel<32, 64>': ("env", {'UNETB200_NO_HALO': '1', 'UNETB200_NO_HALO_WGRAD': '1', 'UNETB200_NO_FIRST_NARROW': '1', 'UNETB200_NO_FIRST_TC': '1'}, (
        'no_halo/wgrad_oihw:bf16:auto:1x32>64x15x17',
    )),
    'narrow_wgrad_kernel<32, 32>': ("env", {'UNETB200_NO_HALO': '1', 'UNETB200_NO_HALO_WGRAD': '1', 'UNETB200_NO_FIRST_NARROW': '1', 'UNETB200_NO_FIRST_TC': '1'}, (
        'no_halo/wgrad_oihw:bf16:auto:1x32>32x14x17',
    )),
    'narrow_wgrad_kernel<32, 16>': ("env", {'UNETB200_NO_HALO': '1', 'UNETB200_NO_HALO_WGRAD': '1', 'UNETB200_NO_FIRST_NARROW': '1', 'UNETB200_NO_FIRST_TC': '1'}, (
        'no_halo/wgrad_oihw:bf16:auto:1x32>16x13x17',
    )),
    'narrow_wgrad_kernel<16, 64>': ("env", {'UNETB200_NO_HALO': '1', 'UNETB200_NO_HALO_WGRAD': '1', 'UNETB200_NO_FIRST_NARROW': '1', 'UNETB200_NO_FIRST_TC': '1'}, (
        'no_halo/wgrad_oihw:bf16:auto:1x16>64x15x16',
    )),
    'narrow_wgrad_kernel<16, 32>': ("env", {'UNETB200_NO_HALO': '1', 'UNETB200_NO_HALO_WGRAD': '1', 'UNETB200_NO_FIRST_NARROW': '1', 'UNETB200_NO_FIRST_TC': '1'}, (
        'no_halo/wgrad_oihw:bf16:auto:1x16>32x14x16',
    )),
    'narrow_wgrad_kernel<16, 16>': ("env", {'UNETB200_NO_HALO': '1', 'UNETB200_NO_HALO_WGRAD': '1', 'UNETB200_NO_FIRST_NARROW': '1', 'UNETB200_NO_FIRST_TC': '1'}, (
        'no_halo/wgrad_oihw:bf16:auto:1x16>16x13x16',
    )),
    'narrow_wgrad_kernel<8, 64>': ("env", {'UNETB200_NO_HALO': '1', 'UNETB200_NO_HALO_WGRAD': '1', 'UNETB200_NO_FIRST_NARROW': '1', 'UNETB200_NO_FIRST_TC': '1'}, (
        'no_halo/wgrad_oihw:bf16:auto:1x8>64x15x15',
    )),
    'narrow_wgrad_kernel<8, 32>': ("env", {'UNETB200_NO_HALO': '1', 'UNETB200_NO_HALO_WGRAD': '1', 'UNETB200_NO_FIRST_NARROW': '1', 'UNETB200_NO_FIRST_TC': '1'}, (
        'no_halo/wgrad_oihw:bf16:auto:1x8>32x14x15',
    )),
    'narrow_wgrad_kernel<8, 16>': ("env", {'UNETB200_NO_HALO': '1', 'UNETB200_NO_HALO_WGRAD': '1', 'UNETB200_NO_FIRST_NARROW': '1', 'UNETB200_NO_FIRST_TC': '1'}, (
        'no_halo/wgrad_oihw:bf16:auto:1x8>16x13x15',
    )),
    'narrow_wgrad_kernel<4, 64>': ("unreachable",
        'narrow_wgrad_supported uses narrow_shape_ok, which rejects C_in <= 4 with N = 64 under every switch; instantiated by the NT = 64 arm of the dispatch'),
    'narrow_wgrad_kernel<4, 32>': ("env", {'UNETB200_NO_HALO': '1', 'UNETB200_NO_HALO_WGRAD': '1', 'UNETB200_NO_FIRST_NARROW': '1', 'UNETB200_NO_FIRST_TC': '1'}, (
        'no_halo/wgrad_oihw:bf16:auto:1x4>32x14x14',
    )),
    'narrow_wgrad_kernel<4, 16>': ("env", {'UNETB200_NO_HALO': '1', 'UNETB200_NO_HALO_WGRAD': '1', 'UNETB200_NO_FIRST_NARROW': '1', 'UNETB200_NO_FIRST_TC': '1'}, (
        'no_halo/wgrad_oihw:bf16:auto:1x4>16x13x14',
    )),
    'narrow_wgrad_kernel<3, 64>': ("unreachable",
        'narrow_wgrad_supported uses narrow_shape_ok, which rejects C_in <= 4 with N = 64 under every switch; instantiated by the NT = 64 arm of the dispatch'),
    'narrow_wgrad_kernel<3, 32>': ("env", {'UNETB200_NO_HALO': '1', 'UNETB200_NO_HALO_WGRAD': '1', 'UNETB200_NO_FIRST_NARROW': '1', 'UNETB200_NO_FIRST_TC': '1'}, (
        'no_halo/wgrad_oihw:bf16:auto:1x3>32x14x13',
    )),
    'narrow_wgrad_kernel<3, 16>': ("env", {'UNETB200_NO_HALO': '1', 'UNETB200_NO_HALO_WGRAD': '1', 'UNETB200_NO_FIRST_NARROW': '1', 'UNETB200_NO_FIRST_TC': '1'}, (
        'no_halo/wgrad_oihw:bf16:auto:1x3>16x13x13',
    )),
    'narrow_wgrad_kernel<2, 64>': ("unreachable",
        'narrow_wgrad_supported uses narrow_shape_ok, which rejects C_in <= 4 with N = 64 under every switch; instantiated by the NT = 64 arm of the dispatch'),
    'narrow_wgrad_kernel<2, 32>': ("env", {'UNETB200_NO_HALO': '1', 'UNETB200_NO_HALO_WGRAD': '1', 'UNETB200_NO_FIRST_NARROW': '1', 'UNETB200_NO_FIRST_TC': '1'}, (
        'no_halo/wgrad_oihw:bf16:auto:1x2>32x14x12',
    )),
    'narrow_wgrad_kernel<2, 16>': ("env", {'UNETB200_NO_HALO': '1', 'UNETB200_NO_HALO_WGRAD': '1', 'UNETB200_NO_FIRST_NARROW': '1', 'UNETB200_NO_FIRST_TC': '1'}, (
        'no_halo/wgrad_oihw:bf16:auto:1x2>16x13x12',
    )),
    'narrow_wgrad_kernel<1, 64>': ("unreachable",
        'narrow_wgrad_supported uses narrow_shape_ok, which rejects C_in <= 4 with N = 64 under every switch; instantiated by the NT = 64 arm of the dispatch'),
    'narrow_wgrad_kernel<1, 32>': ("env", {'UNETB200_NO_HALO': '1', 'UNETB200_NO_HALO_WGRAD': '1', 'UNETB200_NO_FIRST_NARROW': '1', 'UNETB200_NO_FIRST_TC': '1'}, (
        'no_halo/wgrad_oihw:bf16:auto:1x1>32x14x11',
    )),
    'narrow_wgrad_kernel<1, 16>': ("env", {'UNETB200_NO_HALO': '1', 'UNETB200_NO_HALO_WGRAD': '1', 'UNETB200_NO_FIRST_NARROW': '1', 'UNETB200_NO_FIRST_TC': '1'}, (
        'no_halo/wgrad_oihw:bf16:auto:1x1>16x13x11',
    )),
    'narrow_conv_kernel<64, 32, 0>': ("env", {'UNETB200_NO_HALO': '1', 'UNETB200_NO_HALO_WGRAD': '1', 'UNETB200_NO_FIRST_NARROW': '1', 'UNETB200_NO_FIRST_TC': '1'}, (
        'no_halo/fprop:bf16:auto:1x64>32x14x18',
    )),
    'narrow_conv_kernel<64, 16, 0>': ("env", {'UNETB200_NO_HALO': '1', 'UNETB200_NO_HALO_WGRAD': '1', 'UNETB200_NO_FIRST_NARROW': '1', 'UNETB200_NO_FIRST_TC': '1'}, (
        'no_halo/fprop:bf16:auto:1x64>16x13x18',
    )),
    'narrow_conv_kernel<64, 32, 1>': ("env", {'UNETB200_NO_HALO': '1', 'UNETB200_NO_HALO_WGRAD': '1', 'UNETB200_NO_FIRST_NARROW': '1', 'UNETB200_NO_FIRST_TC': '1'}, (
        'no_halo/affine:bf16:auto:1x64>32x14x18',
    )),
    'narrow_conv_kernel<64, 16, 1>': ("env", {'UNETB200_NO_HALO': '1', 'UNETB200_NO_HALO_WGRAD': '1', 'UNETB200_NO_FIRST_NARROW': '1', 'UNETB200_NO_FIRST_TC': '1'}, (
        'no_halo/affine:bf16:auto:1x64>16x13x18',
    )),
    'narrow_conv_kernel<32, 64, 0>': ("env", {'UNETB200_NO_HALO': '1', 'UNETB200_NO_HALO_WGRAD': '1', 'UNETB200_NO_FIRST_NARROW': '1', 'UNETB200_NO_FIRST_TC': '1'}, (
        'no_halo/fprop:bf16:auto:1x32>64x15x17',
    )),
    'narrow_conv_kernel<32, 32, 0>': ("env", {'UNETB200_NO_HALO': '1', 'UNETB200_NO_HALO_WGRAD': '1', 'UNETB200_NO_FIRST_NARROW': '1', 'UNETB200_NO_FIRST_TC': '1'}, (
        'no_halo/fprop:bf16:auto:1x32>32x14x17',
    )),
    'narrow_conv_kernel<32, 16, 0>': ("env", {'UNETB200_NO_HALO': '1', 'UNETB200_NO_HALO_WGRAD': '1', 'UNETB200_NO_FIRST_NARROW': '1', 'UNETB200_NO_FIRST_TC': '1'}, (
        'no_halo/fprop:bf16:auto:1x32>16x13x17',
    )),
    'narrow_conv_kernel<32, 64, 1>': ("env", {'UNETB200_NO_HALO': '1', 'UNETB200_NO_HALO_WGRAD': '1', 'UNETB200_NO_FIRST_NARROW': '1', 'UNETB200_NO_FIRST_TC': '1'}, (
        'no_halo/affine:bf16:auto:1x32>64x15x17',
    )),
    'narrow_conv_kernel<32, 32, 1>': ("env", {'UNETB200_NO_HALO': '1', 'UNETB200_NO_HALO_WGRAD': '1', 'UNETB200_NO_FIRST_NARROW': '1', 'UNETB200_NO_FIRST_TC': '1'}, (
        'no_halo/affine:bf16:auto:1x32>32x14x17',
    )),
    'narrow_conv_kernel<32, 16, 1>': ("env", {'UNETB200_NO_HALO': '1', 'UNETB200_NO_HALO_WGRAD': '1', 'UNETB200_NO_FIRST_NARROW': '1', 'UNETB200_NO_FIRST_TC': '1'}, (
        'no_halo/affine:bf16:auto:1x32>16x13x17',
    )),
    'narrow_conv_kernel<16, 64, 0>': ("env", {'UNETB200_NO_HALO': '1', 'UNETB200_NO_HALO_WGRAD': '1', 'UNETB200_NO_FIRST_NARROW': '1', 'UNETB200_NO_FIRST_TC': '1'}, (
        'no_halo/fprop:bf16:auto:1x16>64x15x16',
    )),
    'narrow_conv_kernel<16, 32, 0>': ("env", {'UNETB200_NO_HALO': '1', 'UNETB200_NO_HALO_WGRAD': '1', 'UNETB200_NO_FIRST_NARROW': '1', 'UNETB200_NO_FIRST_TC': '1'}, (
        'no_halo/fprop:bf16:auto:1x16>32x14x16',
    )),
    'narrow_conv_kernel<16, 16, 0>': ("env", {'UNETB200_NO_HALO': '1', 'UNETB200_NO_HALO_WGRAD': '1', 'UNETB200_NO_FIRST_NARROW': '1', 'UNETB200_NO_FIRST_TC': '1'}, (
        'no_halo/fprop:bf16:auto:1x16>16x13x16',
    )),
    'narrow_conv_kernel<16, 64, 1>': ("env", {'UNETB200_NO_HALO': '1', 'UNETB200_NO_HALO_WGRAD': '1', 'UNETB200_NO_FIRST_NARROW': '1', 'UNETB200_NO_FIRST_TC': '1'}, (
        'no_halo/affine:bf16:auto:1x16>64x15x16',
    )),
    'narrow_conv_kernel<16, 32, 1>': ("env", {'UNETB200_NO_HALO': '1', 'UNETB200_NO_HALO_WGRAD': '1', 'UNETB200_NO_FIRST_NARROW': '1', 'UNETB200_NO_FIRST_TC': '1'}, (
        'no_halo/affine:bf16:auto:1x16>32x14x16',
    )),
    'narrow_conv_kernel<16, 16, 1>': ("env", {'UNETB200_NO_HALO': '1', 'UNETB200_NO_HALO_WGRAD': '1', 'UNETB200_NO_FIRST_NARROW': '1', 'UNETB200_NO_FIRST_TC': '1'}, (
        'no_halo/affine:bf16:auto:1x16>16x13x16',
    )),
    'narrow_conv_kernel<8, 64, 0>': ("env", {'UNETB200_NO_HALO': '1', 'UNETB200_NO_HALO_WGRAD': '1', 'UNETB200_NO_FIRST_NARROW': '1', 'UNETB200_NO_FIRST_TC': '1'}, (
        'no_halo/fprop:bf16:auto:1x8>64x15x15',
    )),
    'narrow_conv_kernel<8, 32, 0>': ("env", {'UNETB200_NO_HALO': '1', 'UNETB200_NO_HALO_WGRAD': '1', 'UNETB200_NO_FIRST_NARROW': '1', 'UNETB200_NO_FIRST_TC': '1'}, (
        'no_halo/fprop:bf16:auto:1x8>32x14x15',
    )),
    'narrow_conv_kernel<8, 16, 0>': ("env", {'UNETB200_NO_HALO': '1', 'UNETB200_NO_HALO_WGRAD': '1', 'UNETB200_NO_FIRST_NARROW': '1', 'UNETB200_NO_FIRST_TC': '1'}, (
        'no_halo/fprop:bf16:auto:1x8>16x13x15',
    )),
    'narrow_conv_kernel<8, 64, 1>': ("env", {'UNETB200_NO_HALO': '1', 'UNETB200_NO_HALO_WGRAD': '1', 'UNETB200_NO_FIRST_NARROW': '1', 'UNETB200_NO_FIRST_TC': '1'}, (
        'no_halo/affine:bf16:auto:1x8>64x15x15',
    )),
    'narrow_conv_kernel<8, 32, 1>': ("env", {'UNETB200_NO_HALO': '1', 'UNETB200_NO_HALO_WGRAD': '1', 'UNETB200_NO_FIRST_NARROW': '1', 'UNETB200_NO_FIRST_TC': '1'}, (
        'no_halo/affine:bf16:auto:1x8>32x14x15',
    )),
    'narrow_conv_kernel<8, 16, 1>': ("env", {'UNETB200_NO_HALO': '1', 'UNETB200_NO_HALO_WGRAD': '1', 'UNETB200_NO_FIRST_NARROW': '1', 'UNETB200_NO_FIRST_TC': '1'}, (
        'no_halo/affine:bf16:auto:1x8>16x13x15',
    )),
    'narrow_conv_kernel<4, 64, 0>': ("unreachable",
        'narrow_shape_ok (conv_narrow.cu) rejects C_in <= 4 with N = 64 under every switch: the first-layer engines own that shape; instantiated by the NT = 64 arm of the dispatch'),
    'narrow_conv_kernel<4, 32, 0>': ("env", {'UNETB200_NO_HALO': '1', 'UNETB200_NO_HALO_WGRAD': '1', 'UNETB200_NO_FIRST_NARROW': '1', 'UNETB200_NO_FIRST_TC': '1'}, (
        'no_halo/fprop:bf16:auto:1x4>32x14x14',
    )),
    'narrow_conv_kernel<4, 16, 0>': ("env", {'UNETB200_NO_HALO': '1', 'UNETB200_NO_HALO_WGRAD': '1', 'UNETB200_NO_FIRST_NARROW': '1', 'UNETB200_NO_FIRST_TC': '1'}, (
        'no_halo/fprop:bf16:auto:1x4>16x13x14',
    )),
    'narrow_conv_kernel<4, 64, 1>': ("unreachable",
        'narrow_shape_ok (conv_narrow.cu) rejects C_in <= 4 with N = 64 under every switch: the first-layer engines own that shape; instantiated by the NT = 64 arm of the dispatch'),
    'narrow_conv_kernel<4, 32, 1>': ("env", {'UNETB200_NO_HALO': '1', 'UNETB200_NO_HALO_WGRAD': '1', 'UNETB200_NO_FIRST_NARROW': '1', 'UNETB200_NO_FIRST_TC': '1'}, (
        'no_halo/affine:bf16:auto:1x4>32x14x14',
    )),
    'narrow_conv_kernel<4, 16, 1>': ("env", {'UNETB200_NO_HALO': '1', 'UNETB200_NO_HALO_WGRAD': '1', 'UNETB200_NO_FIRST_NARROW': '1', 'UNETB200_NO_FIRST_TC': '1'}, (
        'no_halo/affine:bf16:auto:1x4>16x13x14',
    )),
    'narrow_conv_kernel<3, 64, 0>': ("unreachable",
        'narrow_shape_ok (conv_narrow.cu) rejects C_in <= 4 with N = 64 under every switch: the first-layer engines own that shape; instantiated by the NT = 64 arm of the dispatch'),
    'narrow_conv_kernel<3, 32, 0>': ("env", {'UNETB200_NO_HALO': '1', 'UNETB200_NO_HALO_WGRAD': '1', 'UNETB200_NO_FIRST_NARROW': '1', 'UNETB200_NO_FIRST_TC': '1'}, (
        'no_halo/fprop:bf16:auto:1x3>32x14x13',
    )),
    'narrow_conv_kernel<3, 16, 0>': ("env", {'UNETB200_NO_HALO': '1', 'UNETB200_NO_HALO_WGRAD': '1', 'UNETB200_NO_FIRST_NARROW': '1', 'UNETB200_NO_FIRST_TC': '1'}, (
        'no_halo/fprop:bf16:auto:1x3>16x13x13',
    )),
    'narrow_conv_kernel<3, 64, 1>': ("unreachable",
        'narrow_shape_ok (conv_narrow.cu) rejects C_in <= 4 with N = 64 under every switch: the first-layer engines own that shape; instantiated by the NT = 64 arm of the dispatch'),
    'narrow_conv_kernel<3, 32, 1>': ("env", {'UNETB200_NO_HALO': '1', 'UNETB200_NO_HALO_WGRAD': '1', 'UNETB200_NO_FIRST_NARROW': '1', 'UNETB200_NO_FIRST_TC': '1'}, (
        'no_halo/affine:bf16:auto:1x3>32x14x13',
    )),
    'narrow_conv_kernel<3, 16, 1>': ("env", {'UNETB200_NO_HALO': '1', 'UNETB200_NO_HALO_WGRAD': '1', 'UNETB200_NO_FIRST_NARROW': '1', 'UNETB200_NO_FIRST_TC': '1'}, (
        'no_halo/affine:bf16:auto:1x3>16x13x13',
    )),
    'narrow_conv_kernel<2, 64, 0>': ("unreachable",
        'narrow_shape_ok (conv_narrow.cu) rejects C_in <= 4 with N = 64 under every switch: the first-layer engines own that shape; instantiated by the NT = 64 arm of the dispatch'),
    'narrow_conv_kernel<2, 32, 0>': ("env", {'UNETB200_NO_HALO': '1', 'UNETB200_NO_HALO_WGRAD': '1', 'UNETB200_NO_FIRST_NARROW': '1', 'UNETB200_NO_FIRST_TC': '1'}, (
        'no_halo/fprop:bf16:auto:1x2>32x14x12',
    )),
    'narrow_conv_kernel<2, 16, 0>': ("env", {'UNETB200_NO_HALO': '1', 'UNETB200_NO_HALO_WGRAD': '1', 'UNETB200_NO_FIRST_NARROW': '1', 'UNETB200_NO_FIRST_TC': '1'}, (
        'no_halo/fprop:bf16:auto:1x2>16x13x12',
    )),
    'narrow_conv_kernel<2, 64, 1>': ("unreachable",
        'narrow_shape_ok (conv_narrow.cu) rejects C_in <= 4 with N = 64 under every switch: the first-layer engines own that shape; instantiated by the NT = 64 arm of the dispatch'),
    'narrow_conv_kernel<2, 32, 1>': ("env", {'UNETB200_NO_HALO': '1', 'UNETB200_NO_HALO_WGRAD': '1', 'UNETB200_NO_FIRST_NARROW': '1', 'UNETB200_NO_FIRST_TC': '1'}, (
        'no_halo/affine:bf16:auto:1x2>32x14x12',
    )),
    'narrow_conv_kernel<2, 16, 1>': ("env", {'UNETB200_NO_HALO': '1', 'UNETB200_NO_HALO_WGRAD': '1', 'UNETB200_NO_FIRST_NARROW': '1', 'UNETB200_NO_FIRST_TC': '1'}, (
        'no_halo/affine:bf16:auto:1x2>16x13x12',
    )),
    'narrow_conv_kernel<1, 64, 0>': ("unreachable",
        'narrow_shape_ok (conv_narrow.cu) rejects C_in <= 4 with N = 64 under every switch: the first-layer engines own that shape; instantiated by the NT = 64 arm of the dispatch'),
    'narrow_conv_kernel<1, 32, 0>': ("env", {'UNETB200_NO_HALO': '1', 'UNETB200_NO_HALO_WGRAD': '1', 'UNETB200_NO_FIRST_NARROW': '1', 'UNETB200_NO_FIRST_TC': '1'}, (
        'no_halo/fprop:bf16:auto:1x1>32x14x11',
    )),
    'narrow_conv_kernel<1, 16, 0>': ("env", {'UNETB200_NO_HALO': '1', 'UNETB200_NO_HALO_WGRAD': '1', 'UNETB200_NO_FIRST_NARROW': '1', 'UNETB200_NO_FIRST_TC': '1'}, (
        'no_halo/fprop:bf16:auto:1x1>16x13x11',
    )),
    'narrow_conv_kernel<1, 64, 1>': ("unreachable",
        'narrow_shape_ok (conv_narrow.cu) rejects C_in <= 4 with N = 64 under every switch: the first-layer engines own that shape; instantiated by the NT = 64 arm of the dispatch'),
    'narrow_conv_kernel<1, 32, 1>': ("env", {'UNETB200_NO_HALO': '1', 'UNETB200_NO_HALO_WGRAD': '1', 'UNETB200_NO_FIRST_NARROW': '1', 'UNETB200_NO_FIRST_TC': '1'}, (
        'no_halo/affine:bf16:auto:1x1>32x14x11',
    )),
    'narrow_conv_kernel<1, 16, 1>': ("env", {'UNETB200_NO_HALO': '1', 'UNETB200_NO_HALO_WGRAD': '1', 'UNETB200_NO_FIRST_NARROW': '1', 'UNETB200_NO_FIRST_TC': '1'}, (
        'no_halo/affine:bf16:auto:1x1>16x13x11',
    )),
    'pack_multi_kernel<float>': (
        'pack_multi:fp32:f3',
    ),
    'pack_multi_kernel<__nv_bfloat16>': (
        'pack_multi:bf16:f3',
    ),
    'pack_weights_kernel<float>': (
        'pack_single:fp32:d3',
    ),
    'pack_weights_kernel<__nv_bfloat16>': (
        'pack_single:bf16:d3',
    ),
    'pack_weights_t_kernel<float>': (
        'pack_single:fp32:d3_cl',
    ),
    'pack_weights_t_kernel<__nv_bfloat16>': (
        'pack_single:bf16:d3_cl',
    ),
    'gconv_wgrad_simt_kernel<float, false, 64>': (
        'wgrad_oihw:fp32:simt:2x6>80x9x11',
    ),
    'gconv_wgrad_simt_kernel<float, false, 32>': (
        'wgrad_oihw:fp32:simt:1x2>32x12x16',
        'wgrad_oihw:fp32:simt:1x3>32x12x16',
        'wgrad_oihw:fp32:simt:2x6>24x9x11',
    ),
    'gconv_wgrad_simt_kernel<float, false, 16>': (
        'wgrad_oihw:fp32:simt:2x6>12x9x11',
    ),
    'gconv_wgrad_simt_kernel<float, true, 64>': (
        'convT_wgrad:fp32:simt:2x32>16x4x5_pad12',
        'wgrad_oihw:fp32:simt:1x64>64x8x8_slice',
        'wgrad_oihw:fp32:simt:2x48>80x9x11',
    ),
    'gconv_wgrad_simt_kernel<float, true, 32>': (
        'wgrad_oihw:fp32:simt:1x4>32x12x16',
        'wgrad_oihw:fp32:simt:2x48>24x9x11',
    ),
    'gconv_wgrad_simt_kernel<float, true, 16>': (
        'wgrad_oihw:fp32:simt:2x48>12x9x11',
    ),
    'gconv_wgrad_simt_kernel<__nv_bfloat16, false, 64>': (
        'wgrad_oihw:bf16:auto:2x2>64x30x34',
        'wgrad_oihw:bf16:auto:2x3>64x30x34',
        'wgrad_oihw:bf16:simt:2x6>80x9x11',
    ),
    'gconv_wgrad_simt_kernel<__nv_bfloat16, false, 32>': (
        'wgrad_oihw:bf16:simt:1x2>32x12x16',
        'wgrad_oihw:bf16:simt:1x3>32x12x16',
        'wgrad_oihw:bf16:simt:2x6>24x9x11',
    ),
    'gconv_wgrad_simt_kernel<__nv_bfloat16, false, 16>': (
        'wgrad_oihw:bf16:simt:2x6>12x9x11',
    ),
    'gconv_wgrad_simt_kernel<__nv_bfloat16, true, 64>': (
        'convT_wgrad:bf16:simt:2x32>16x4x5_pad12',
        'wgrad_oihw:bf16:auto:2x4>64x30x34',
        'wgrad_oihw:bf16:simt:1x64>64x8x8_slice',
        'wgrad_oihw:bf16:simt:2x48>80x9x11',
    ),
    'gconv_wgrad_simt_kernel<__nv_bfloat16, true, 32>': (
        'wgrad_oihw:bf16:simt:1x4>32x12x16',
        'wgrad_oihw:bf16:simt:2x48>24x9x11',
    ),
    'gconv_wgrad_simt_kernel<__nv_bfloat16, true, 16>': (
        'wgrad_oihw:bf16:simt:2x48>12x9x11',
    ),
    'gconv_fprop_simt_kernel<float, false, 64>': (
        'fprop:fp32:simt:2x6>80x9x11',
    ),
    'gconv_fprop_simt_kernel<float, false, 32>': (
        'fprop:fp32:simt:2x6>24x9x11',
    ),
    'gconv_fprop_simt_kernel<float, false, 16>': (
        'fprop:fp32:simt:2x6>12x9x11',
    ),
    'gconv_fprop_simt_kernel<float, true, 64>': (
        'convT_fprop:fp32:simt:2x32>16x4x5_pad12',
        'dgrad:fp32:simt:1x64>64x8x8_slice',
        'fprop:fp32:simt:1x64>64x8x8_slice',
        'fprop:fp32:simt:2x48>80x9x11',
    ),
    'gconv_fprop_simt_kernel<float, true, 32>': (
        'convT_dgrad:fp32:simt:2x32>16x4x5_pad12',
        'fprop:fp32:simt:2x48>24x9x11',
    ),
    'gconv_fprop_simt_kernel<float, true, 16>': (
        'fprop:fp32:simt:2x48>12x9x11',
    ),
    'gconv_fprop_simt_kernel<__nv_bfloat16, false, 64>': (
        'fprop:bf16:simt:2x6>80x9x11',
    ),
    'gconv_fprop_simt_kernel<__nv_bfloat16, false, 32>': (
        'fprop:bf16:simt:2x6>24x9x11',
    ),
    'gconv_fprop_simt_kernel<__nv_bfloat16, false, 16>': (
        'fprop:bf16:simt:2x6>12x9x11',
    ),
    'gconv_fprop_simt_kernel<__nv_bfloat16, true, 64>': (
        'convT_fprop:bf16:simt:2x32>16x4x5_pad12',
        'dgrad:bf16:simt:1x64>64x8x8_slice',
        'fprop:bf16:simt:1x64>64x8x8_slice',
        'fprop:bf16:simt:2x48>80x9x11',
    ),
    'gconv_fprop_simt_kernel<__nv_bfloat16, true, 32>': (
        'convT_dgrad:bf16:simt:2x32>16x4x5_pad12',
        'fprop:bf16:simt:2x48>24x9x11',
    ),
    'gconv_fprop_simt_kernel<__nv_bfloat16, true, 16>': (
        'fprop:bf16:simt:2x48>12x9x11',
    ),
    'wgrad_reduce_t_kernel<8>': (
        'wgrad_cl:bf16:tc:2x64>64x64x64',
    ),
    'wgrad_reduce_t_kernel<32>': (
        'wgrad_cl:bf16:tc:2x64>64x128x128',
    ),
    'wgrad_reduce_multi_kernel': (
        'wgrad_multi:bf16:tc:2x128>128x20x28',
    ),
    'wgrad_reduce_t4_kernel': (
        'wgrad_cl:bf16:tc:1x128>64x40x36',
        'wgrad_cl:bf16:tc:1x256>256x12x10',
        'wgrad_cl:bf16:tc:2x128>128x32x48',
        'wgrad_cl:bf16:tc:2x128>64x24x20',
        'wgrad_cl:bf16:tc:3x512>256x16x8',
        'wgrad_cl:fp32:tc:2x128>128x10x12',
    ),
    'wgrad_reduce_kernel': (
        'convT_wgrad:bf16:simt:2x32>16x4x5_pad12',
        'convT_wgrad:bf16:tc:1x16>8x9x7',
        'convT_wgrad:bf16:tc:1x256>128x5x4_pad11',
        'convT_wgrad:bf16:tc:1x32>32x11x9',
        'convT_wgrad:bf16:tc:1x512>256x4x4',
        'convT_wgrad:bf16:tc:1x64>32x13x11',
        'convT_wgrad:bf16:tc:2x128>128x9x7_pad10',
        'convT_wgrad:bf16:tc:2x128>64x6x10',
        'convT_wgrad:bf16:tc:2x32>16x10x8',
        'convT_wgrad:bf16:tc:2x64>16x12x10',
        'convT_wgrad:bf16:tc:2x64>64x7x9',
        'convT_wgrad:fp32:simt:2x32>16x4x5_pad12',
        'convT_wgrad:fp32:tc:1x128>64x4x4_pad10',
        'convT_wgrad:fp32:tc:1x256>128x5x6_pad01',
        'convT_wgrad:fp32:tc:2x64>64x6x5',
        'wgrad_oihw:bf16:auto:1x16>32x33x20',
        'wgrad_oihw:bf16:auto:1x16>8x20x24',
        'wgrad_oihw:bf16:auto:1x32>16x33x20',
        'wgrad_oihw:bf16:auto:1x32>64x33x20',
        'wgrad_oihw:bf16:auto:1x64>32x33x20',
        'wgrad_oihw:bf16:auto:2x16>16x24x17',
        'wgrad_oihw:bf16:auto:2x16>64x24x17',
        'wgrad_oihw:bf16:auto:2x1>16x37x45',
        'wgrad_oihw:bf16:auto:2x1>32x37x45',
        'wgrad_oihw:bf16:auto:2x1>64x30x34',
        'wgrad_oihw:bf16:auto:2x1>8x37x45',
        'wgrad_oihw:bf16:auto:2x2>64x30x34',
        'wgrad_oihw:bf16:auto:2x32>32x16x16_slice',
        'wgrad_oihw:bf16:auto:2x32>32x24x17',
        'wgrad_oihw:bf16:auto:2x3>64x30x34',
        'wgrad_oihw:bf16:auto:2x4>64x30x34',
        'wgrad_oihw:bf16:auto:2x64>16x24x17',
        'wgrad_oihw:bf16:auto:2x8>8x37x41',
        'wgrad_oihw:bf16:auto:8x16>16x128x128',
        'wgrad_oihw:bf16:simt:1x1>128x9x13',
        'wgrad_oihw:bf16:simt:1x2>32x12x16',
        'wgrad_oihw:bf16:simt:1x3>32x12x16',
        'wgrad_oihw:bf16:simt:1x4>32x12x16',
        'wgrad_oihw:bf16:simt:1x64>64x8x8_slice',
        'wgrad_oihw:bf16:simt:2x1>64x20x22',
        'wgrad_oihw:bf16:simt:2x48>12x9x11',
        'wgrad_oihw:bf16:simt:2x48>24x9x11',
        'wgrad_oihw:bf16:simt:2x48>80x9x11',
        'wgrad_oihw:bf16:simt:2x6>12x9x11',
        'wgrad_oihw:bf16:simt:2x6>24x9x11',
        'wgrad_oihw:bf16:simt:2x6>80x9x11',
        'wgrad_oihw:bf16:tc:1x128>64x40x36',
        'wgrad_oihw:bf16:tc:1x256>256x12x10',
        'wgrad_oihw:bf16:tc:1x64>128x17x21_slice',
        'wgrad_oihw:bf16:tc:1x64>64x33x17',
        'wgrad_oihw:bf16:tc:2x128>128x20x28',
        'wgrad_oihw:bf16:tc:2x128>128x32x48',
        'wgrad_oihw:bf16:tc:2x128>64x24x20',
        'wgrad_oihw:bf16:tc:2x64>64x64x64',
        'wgrad_oihw:bf16:tc:3x512>256x16x8',
        'wgrad_oihw:fp32:simt:1x16>16x17x23',
        'wgrad_oihw:fp32:simt:1x16>32x17x23',
        'wgrad_oihw:fp32:simt:1x16>64x17x23',
        'wgrad_oihw:fp32:simt:1x1>128x9x13',
        'wgrad_oihw:fp32:simt:1x2>32x12x16',
        'wgrad_oihw:fp32:simt:1x32>16x17x23',
        'wgrad_oihw:fp32:simt:1x32>32x17x23',
        'wgrad_oihw:fp32:simt:1x32>64x17x23',
        'wgrad_oihw:fp32:simt:1x3>32x12x16',
        'wgrad_oihw:fp32:simt:1x4>32x12x16',
        'wgrad_oihw:fp32:simt:1x64>16x17x23',
        'wgrad_oihw:fp32:simt:1x64>32x17x23',
        'wgrad_oihw:fp32:simt:1x64>64x8x8_slice',
        'wgrad_oihw:fp32:simt:2x16>8x13x19',
        'wgrad_oihw:fp32:simt:2x1>64x20x22',
        'wgrad_oihw:fp32:simt:2x32>8x13x19',
        'wgrad_oihw:fp32:simt:2x48>12x9x11',
        'wgrad_oihw:fp32:simt:2x48>24x9x11',
        'wgrad_oihw:fp32:simt:2x48>80x9x11',
        'wgrad_oihw:fp32:simt:2x64>8x13x19',
        'wgrad_oihw:fp32:simt:2x6>12x9x11',
        'wgrad_oihw:fp32:simt:2x6>24x9x11',
        'wgrad_oihw:fp32:simt:2x6>80x9x11',
        'wgrad_oihw:fp32:simt:2x8>16x13x19',
        'wgrad_oihw:fp32:simt:2x8>32x13x19',
        'wgrad_oihw:fp32:simt:2x8>64x13x19',
        'wgrad_oihw:fp32:simt:2x8>8x13x19',
        'wgrad_oihw:fp32:tc:1x64>64x19x21',
        'wgrad_oihw:fp32:tc:2x128>128x10x12',
        'wgrad_oihw:fp32:tc:2x64>128x12x12',
        'no_halo/wgrad_oihw:bf16:auto:1x16>16x13x16',
        'no_halo/wgrad_oihw:bf16:auto:1x16>32x14x16',
        'no_halo/wgrad_oihw:bf16:auto:1x16>64x15x16',
        'no_halo/wgrad_oihw:bf16:auto:1x1>16x13x11',
        'no_halo/wgrad_oihw:bf16:auto:1x1>32x14x11',
        'no_halo/wgrad_oihw:bf16:auto:1x2>16x13x12',
        'no_halo/wgrad_oihw:bf16:auto:1x2>32x14x12',
        'no_halo/wgrad_oihw:bf16:auto:1x32>16x13x17',
        'no_halo/wgrad_oihw:bf16:auto:1x32>32x14x17',
        'no_halo/wgrad_oihw:bf16:auto:1x32>64x15x17',
        'no_halo/wgrad_oihw:bf16:auto:1x3>16x13x13',
        'no_halo/wgrad_oihw:bf16:auto:1x3>32x14x13',
        'no_halo/wgrad_oihw:bf16:auto:1x4>16x13x14',
        'no_halo/wgrad_oihw:bf16:auto:1x4>32x14x14',
        'no_halo/wgrad_oihw:bf16:auto:1x64>16x13x18',
        'no_halo/wgrad_oihw:bf16:auto:1x64>32x14x18',
        'no_halo/wgrad_oihw:bf16:auto:1x8>16x13x15',
        'no_halo/wgrad_oihw:bf16:auto:1x8>32x14x15',
        'no_halo/wgrad_oihw:bf16:auto:1x8>64x15x15',
        'tc3w_stages5/wgrad_oihw:bf16:tc:1x256>256x12x10',
        'tc4w_all/wgrad_oihw:bf16:tc:1x256>256x12x10',
    ),
    'stats_reduce_kernel': (
        'dgrad_bnbwd:bf16:auto:2x16>16x18x22',
        'dgrad_bnbwd:bf16:auto:2x16>32x18x22',
        'dgrad_bnbwd:bf16:auto:2x16>64x18x22',
        'dgrad_bnbwd:bf16:auto:2x32>16x18x22',
        'dgrad_bnbwd:bf16:auto:2x32>32x18x22',
        'dgrad_bnbwd:bf16:auto:2x32>64x18x22',
        'dgrad_bnbwd:bf16:auto:2x8>8x37x41',
        'fprop:bf16:auto:1x16>32x33x20',
        'fprop:bf16:auto:1x16>8x20x24',
        'fprop:bf16:auto:1x32>16x33x20',
        'fprop:bf16:auto:1x32>64x33x20',
        'fprop:bf16:auto:1x64>32x33x20',
        'fprop:bf16:auto:2x16>16x24x17',
        'fprop:bf16:auto:2x16>64x24x17',
        'fprop:bf16:auto:2x1>16x37x45',
        'fprop:bf16:auto:2x1>32x37x45',
        'fprop:bf16:auto:2x1>64x30x34',
        'fprop:bf16:auto:2x1>8x37x45',
        'fprop:bf16:auto:2x2>64x30x34',
        'fprop:bf16:auto:2x32>32x16x16_slice',
        'fprop:bf16:auto:2x32>32x24x17',
        'fprop:bf16:auto:2x3>64x30x34',
        'fprop:bf16:auto:2x4>64x30x34',
        'fprop:bf16:auto:2x64>16x24x17',
        'fprop:bf16:auto:2x8>8x37x41',
        'fprop:bf16:auto:8x16>16x128x128',
        'fprop:bf16:simt:1x1>128x9x13',
        'fprop:bf16:simt:1x2>32x11x13',
        'fprop:bf16:simt:1x2>32x12x16',
        'fprop:bf16:simt:1x3>32x11x13',
        'fprop:bf16:simt:1x3>32x12x16',
        'fprop:bf16:simt:1x4>32x11x13',
        'fprop:bf16:simt:1x4>32x12x16',
        'fprop:bf16:simt:1x64>64x8x8_slice',
        'fprop:bf16:simt:2x1>64x20x22',
        'fprop:bf16:simt:2x48>12x9x11',
        'fprop:bf16:simt:2x48>24x9x11',
        'fprop:bf16:simt:2x48>80x9x11',
        'fprop:bf16:simt:2x6>12x9x11',
        'fprop:bf16:simt:2x6>24x9x11',
        'fprop:bf16:simt:2x6>80x9x11',
        'fprop:fp32:prefer:1x16>16x21x19',
        'fprop:fp32:prefer:1x16>32x21x19',
        'fprop:fp32:prefer:1x32>16x21x19',
        'fprop:fp32:prefer:1x32>32x21x19',
        'fprop:fp32:simt:1x16>16x17x23',
        'fprop:fp32:simt:1x16>32x17x23',
        'fprop:fp32:simt:1x16>64x17x23',
        'fprop:fp32:simt:1x1>128x9x13',
        'fprop:fp32:simt:1x2>32x11x13',
        'fprop:fp32:simt:1x2>32x12x16',
        'fprop:fp32:simt:1x32>16x17x23',
        'fprop:fp32:simt:1x32>32x17x23',
        'fprop:fp32:simt:1x32>64x17x23',
        'fprop:fp32:simt:1x3>32x11x13',
        'fprop:fp32:simt:1x3>32x12x16',
        'fprop:fp32:simt:1x4>32x11x13',
        'fprop:fp32:simt:1x4>32x12x16',
        'fprop:fp32:simt:1x64>16x17x23',
        'fprop:fp32:simt:1x64>32x17x23',
        'fprop:fp32:simt:1x64>64x8x8_slice',
        'fprop:fp32:simt:2x1>64x20x22',
        'fprop:fp32:simt:2x48>12x9x11',
        'fprop:fp32:simt:2x48>24x9x11',
        'fprop:fp32:simt:2x48>80x9x11',
        'fprop:fp32:simt:2x6>12x9x11',
        'fprop:fp32:simt:2x6>24x9x11',
        'fprop:fp32:simt:2x6>80x9x11',
        'no_halo/fprop:bf16:auto:1x16>16x13x16',
        'no_halo/fprop:bf16:auto:1x16>32x14x16',
        'no_halo/fprop:bf16:auto:1x16>64x15x16',
        'no_halo/fprop:bf16:auto:1x1>16x13x11',
        'no_halo/fprop:bf16:auto:1x1>32x14x11',
        'no_halo/fprop:bf16:auto:1x2>16x13x12',
        'no_halo/fprop:bf16:auto:1x2>32x14x12',
        'no_halo/fprop:bf16:auto:1x32>16x13x17',
        'no_halo/fprop:bf16:auto:1x32>32x14x17',
        'no_halo/fprop:bf16:auto:1x32>64x15x17',
        'no_halo/fprop:bf16:auto:1x3>16x13x13',
        'no_halo/fprop:bf16:auto:1x3>32x14x13',
        'no_halo/fprop:bf16:auto:1x4>16x13x14',
        'no_halo/fprop:bf16:auto:1x4>32x14x14',
        'no_halo/fprop:bf16:auto:1x64>16x13x18',
        'no_halo/fprop:bf16:auto:1x64>32x14x18',
        'no_halo/fprop:bf16:auto:1x8>16x13x15',
        'no_halo/fprop:bf16:auto:1x8>32x14x15',
        'no_halo/fprop:bf16:auto:1x8>64x15x15',
        'no_halo/fprop:bf16:simt:2x1>64x20x22',
    ),
    'fprop_narrow_f32_kernel<64, 32>': (
        'fprop:fp32:simt:1x64>32x17x23',
    ),
    'fprop_narrow_f32_kernel<64, 16>': (
        'fprop:fp32:simt:1x64>16x17x23',
    ),
    'fprop_narrow_f32_kernel<32, 64>': (
        'fprop:fp32:simt:1x32>64x17x23',
    ),
    'fprop_narrow_f32_kernel<32, 32>': (
        'fprop:fp32:simt:1x32>32x17x23',
    ),
    'fprop_narrow_f32_kernel<32, 16>': (
        'fprop:fp32:simt:1x32>16x17x23',
    ),
    'fprop_narrow_f32_kernel<16, 64>': (
        'fprop:fp32:simt:1x16>64x17x23',
    ),
    'fprop_narrow_f32_kernel<16, 32>': (
        'fprop:fp32:simt:1x16>32x17x23',
    ),
    'fprop_narrow_f32_kernel<16, 16>': (
        'fprop:fp32:simt:1x16>16x17x23',
    ),
    'wgrad_narrow_f32_kernel<64, 8>': (
        'wgrad_oihw:fp32:simt:2x64>8x13x19',
    ),
    'wgrad_narrow_f32_kernel<32, 8>': (
        'wgrad_oihw:fp32:simt:2x32>8x13x19',
    ),
    'wgrad_narrow_f32_kernel<16, 8>': (
        'wgrad_oihw:fp32:simt:2x16>8x13x19',
    ),
    'wgrad_narrow_f32_kernel<8, 64>': (
        'wgrad_oihw:fp32:simt:2x8>64x13x19',
    ),
    'wgrad_narrow_f32_kernel<8, 32>': (
        'wgrad_oihw:fp32:simt:2x8>32x13x19',
    ),
    'wgrad_narrow_f32_kernel<8, 16>': (
        'wgrad_oihw:fp32:simt:2x8>16x13x19',
    ),
    'wgrad_narrow_f32_kernel<8, 8>': (
        'wgrad_oihw:fp32:simt:2x8>8x13x19',
    ),
    'wgrad_narrow_f32_kernel<64, 32>': (
        'wgrad_oihw:fp32:simt:1x64>32x17x23',
    ),
    'wgrad_narrow_f32_kernel<64, 16>': (
        'wgrad_oihw:fp32:simt:1x64>16x17x23',
    ),
    'wgrad_narrow_f32_kernel<32, 64>': (
        'wgrad_oihw:fp32:simt:1x32>64x17x23',
    ),
    'wgrad_narrow_f32_kernel<32, 32>': (
        'wgrad_oihw:fp32:simt:1x32>32x17x23',
    ),
    'wgrad_narrow_f32_kernel<32, 16>': (
        'wgrad_oihw:fp32:simt:1x32>16x17x23',
    ),
    'wgrad_narrow_f32_kernel<16, 64>': (
        'wgrad_oihw:fp32:simt:1x16>64x17x23',
    ),
    'wgrad_narrow_f32_kernel<16, 32>': (
        'wgrad_oihw:fp32:simt:1x16>32x17x23',
    ),
    'wgrad_narrow_f32_kernel<16, 16>': (
        'wgrad_oihw:fp32:simt:1x16>16x17x23',
    ),
    'first_conv_wgrad_kernel<float>': (
        'wgrad_oihw:fp32:simt:1x1>128x9x13',
    ),
    'first_conv_wgrad_kernel<__nv_bfloat16>': (
        'wgrad_oihw:bf16:simt:1x1>128x9x13',
    ),
    'first_conv_wgrad_tiled_kernel<float>': (
        'wgrad_oihw:fp32:simt:2x1>64x20x22',
    ),
    'first_conv_wgrad_tiled_kernel<__nv_bfloat16>': (
        'wgrad_oihw:bf16:auto:2x1>64x30x34',
        'wgrad_oihw:bf16:simt:2x1>64x20x22',
    ),
    'first_conv_fprop_kernel<float, 4>': (
        'fprop:fp32:simt:1x4>32x11x13',
    ),
    'first_conv_fprop_kernel<float, 3>': (
        'fprop:fp32:simt:1x3>32x11x13',
    ),
    'first_conv_fprop_kernel<float, 2>': (
        'fprop:fp32:simt:1x2>32x11x13',
    ),
    'first_conv_fprop_kernel<float, 1>': (
        'fprop:fp32:simt:1x1>128x9x13',
    ),
    'first_conv_fprop_kernel<__nv_bfloat16, 4>': (
        'fprop:bf16:simt:1x4>32x11x13',
    ),
    'first_conv_fprop_kernel<__nv_bfloat16, 3>': (
        'fprop:bf16:simt:1x3>32x11x13',
    ),
    'first_conv_fprop_kernel<__nv_bfloat16, 2>': (
        'fprop:bf16:simt:1x2>32x11x13',
    ),
    'first_conv_fprop_kernel<__nv_bfloat16, 1>': (
        'fprop:bf16:simt:1x1>128x9x13',
    ),
    'first_conv_fprop_px4_kernel<float, 4>': (
        'fprop:fp32:simt:1x4>32x12x16',
    ),
    'first_conv_fprop_px4_kernel<float, 3>': (
        'fprop:fp32:simt:1x3>32x12x16',
    ),
    'first_conv_fprop_px4_kernel<float, 2>': (
        'fprop:fp32:simt:1x2>32x12x16',
    ),
    'first_conv_fprop_px4_kernel<__nv_bfloat16, 4>': (
        'fprop:bf16:simt:1x4>32x12x16',
    ),
    'first_conv_fprop_px4_kernel<__nv_bfloat16, 3>': (
        'fprop:bf16:simt:1x3>32x12x16',
    ),
    'first_conv_fprop_px4_kernel<__nv_bfloat16, 2>': (
        'fprop:bf16:simt:1x2>32x12x16',
    ),
    'first_conv_fprop_tiled_kernel<float>': (
        'fprop:fp32:simt:2x1>64x20x22',
    ),
    'first_conv_fprop_tiled_kernel<__nv_bfloat16>': ("env", {'UNETB200_NO_HALO': '1', 'UNETB200_NO_HALO_WGRAD': '1', 'UNETB200_NO_FIRST_NARROW': '1', 'UNETB200_NO_FIRST_TC': '1'}, (
        'no_halo/fprop:bf16:simt:2x1>64x20x22',
    )),
    'outconv_bwd_vec_kernel<float, 8, false>': (
        'outconv_bwd:fp32:1x16>8x18x15',
    ),
    'outconv_bwd_vec_kernel<float, 8, true>': (
        'outconv_bwd_bnbwd:fp32:1x16>8x18x15',
    ),
    'outconv_bwd_vec_kernel<float, 7, false>': (
        'outconv_bwd:fp32:2x64>7x17x14',
    ),
    'outconv_bwd_vec_kernel<float, 7, true>': (
        'outconv_bwd_bnbwd:fp32:2x64>7x17x14',
    ),
    'outconv_bwd_vec_kernel<float, 6, false>': (
        'outconv_bwd:fp32:1x16>6x16x13',
    ),
    'outconv_bwd_vec_kernel<float, 6, true>': (
        'outconv_bwd_bnbwd:fp32:1x16>6x16x13',
    ),
    'outconv_bwd_vec_kernel<float, 5, false>': (
        'outconv_bwd:fp32:2x64>5x15x12',
    ),
    'outconv_bwd_vec_kernel<float, 5, true>': (
        'outconv_bwd_bnbwd:fp32:2x64>5x15x12',
    ),
    'outconv_bwd_vec_kernel<float, 4, false>': (
        'outconv_bwd:fp32:1x16>4x14x11',
    ),
    'outconv_bwd_vec_kernel<float, 4, true>': (
        'outconv_bwd_bnbwd:fp32:1x16>4x14x11',
    ),
    'outconv_bwd_vec_kernel<float, 3, false>': (
        'outconv_bwd:fp32:2x64>3x13x10',
    ),
    'outconv_bwd_vec_kernel<float, 3, true>': (
        'outconv_bwd_bnbwd:fp32:2x64>3x13x10',
    ),
    'outconv_bwd_vec_kernel<float, 2, false>': (
        'outconv_bwd:fp32:1x16>2x12x9',
    ),
    'outconv_bwd_vec_kernel<float, 2, true>': (
        'outconv_bwd_bnbwd:fp32:1x16>2x12x9',
    ),
    'outconv_bwd_vec_kernel<float, 1, false>': (
        'outconv_bwd:fp32:2x64>1x11x8',
    ),
    'outconv_bwd_vec_kernel<float, 1, true>': (
        'outconv_bwd_bnbwd:fp32:2x64>1x11x8',
    ),
    'outconv_bwd_scalar_kernel<float>': (
        'outconv_bwd:fp32:1x6>3x7x9',
    ),
    'outconv_bwd_vec_kernel<__nv_bfloat16, 8, false>': (
        'outconv_bwd:bf16:1x16>8x18x15',
    ),
    'outconv_bwd_vec_kernel<__nv_bfloat16, 8, true>': (
        'outconv_bwd_bnbwd:bf16:1x16>8x18x15',
    ),
    'outconv_bwd_vec_kernel<__nv_bfloat16, 7, false>': (
        'outconv_bwd:bf16:2x64>7x17x14',
    ),
    'outconv_bwd_vec_kernel<__nv_bfloat16, 7, true>': (
        'outconv_bwd_bnbwd:bf16:2x64>7x17x14',
    ),
    'outconv_bwd_vec_kernel<__nv_bfloat16, 6, false>': (
        'outconv_bwd:bf16:1x16>6x16x13',
    ),
    'outconv_bwd_vec_kernel<__nv_bfloat16, 6, true>': (
        'outconv_bwd_bnbwd:bf16:1x16>6x16x13',
    ),
    'outconv_bwd_vec_kernel<__nv_bfloat16, 5, false>': (
        'outconv_bwd:bf16:2x64>5x15x12',
    ),
    'outconv_bwd_vec_kernel<__nv_bfloat16, 5, true>': (
        'outconv_bwd_bnbwd:bf16:2x64>5x15x12',
    ),
    'outconv_bwd_vec_kernel<__nv_bfloat16, 4, false>': (
        'outconv_bwd:bf16:1x16>4x14x11',
    ),
    'outconv_bwd_vec_kernel<__nv_bfloat16, 4, true>': (
        'outconv_bwd_bnbwd:bf16:1x16>4x14x11',
    ),
    'outconv_bwd_vec_kernel<__nv_bfloat16, 3, false>': (
        'outconv_bwd:bf16:2x64>3x13x10',
    ),
    'outconv_bwd_vec_kernel<__nv_bfloat16, 3, true>': (
        'outconv_bwd_bnbwd:bf16:2x64>3x13x10',
    ),
    'outconv_bwd_vec_kernel<__nv_bfloat16, 2, false>': (
        'outconv_bwd:bf16:1x16>2x12x9',
    ),
    'outconv_bwd_vec_kernel<__nv_bfloat16, 2, true>': (
        'outconv_bwd_bnbwd:bf16:1x16>2x12x9',
    ),
    'outconv_bwd_vec_kernel<__nv_bfloat16, 1, false>': (
        'outconv_bwd:bf16:2x64>1x11x8',
    ),
    'outconv_bwd_vec_kernel<__nv_bfloat16, 1, true>': (
        'outconv_bwd_bnbwd:bf16:2x64>1x11x8',
    ),
    'outconv_bwd_scalar_kernel<__nv_bfloat16>': (
        'outconv_bwd:bf16:1x6>3x7x9',
    ),
    'outconv_fwd_vec_kernel<float, 8>': (
        'outconv_fwd:fp32:1x16>8x17x15',
    ),
    'outconv_fwd_vec_kernel<float, 7>': (
        'outconv_fwd:fp32:2x64>7x16x14',
    ),
    'outconv_fwd_vec_kernel<float, 6>': (
        'outconv_fwd:fp32:1x16>6x15x13',
    ),
    'outconv_fwd_vec_kernel<float, 5>': (
        'outconv_fwd:fp32:2x64>5x14x12',
    ),
    'outconv_fwd_vec_kernel<float, 4>': (
        'outconv_fwd:fp32:1x16>4x13x11',
    ),
    'outconv_fwd_vec_kernel<float, 3>': (
        'outconv_fwd:fp32:2x64>3x12x10',
    ),
    'outconv_fwd_vec_kernel<float, 2>': (
        'outconv_fwd:fp32:1x16>2x11x9',
    ),
    'outconv_fwd_vec_kernel<float, 1>': (
        'outconv_fwd:fp32:2x64>1x10x8',
    ),
    'outconv_fwd_scalar_kernel<float>': (
        'outconv_fwd:fp32:1x6>3x7x9',
    ),
    'outconv_fwd_vec_kernel<__nv_bfloat16, 8>': (
        'outconv_fwd:bf16:1x16>8x17x15',
    ),
    'outconv_fwd_vec_kernel<__nv_bfloat16, 7>': (
        'outconv_fwd:bf16:2x64>7x16x14',
    ),
    'outconv_fwd_vec_kernel<__nv_bfloat16, 6>': (
        'outconv_fwd:bf16:1x16>6x15x13',
    ),
    'outconv_fwd_vec_kernel<__nv_bfloat16, 5>': (
        'outconv_fwd:bf16:2x64>5x14x12',
    ),
    'outconv_fwd_vec_kernel<__nv_bfloat16, 4>': (
        'outconv_fwd:bf16:1x16>4x13x11',
    ),
    'outconv_fwd_vec_kernel<__nv_bfloat16, 3>': (
        'outconv_fwd:bf16:2x64>3x12x10',
    ),
    'outconv_fwd_vec_kernel<__nv_bfloat16, 2>': (
        'outconv_fwd:bf16:1x16>2x11x9',
    ),
    'outconv_fwd_vec_kernel<__nv_bfloat16, 1>': (
        'outconv_fwd:bf16:2x64>1x10x8',
    ),
    'outconv_fwd_scalar_kernel<__nv_bfloat16>': (
        'outconv_fwd:bf16:1x6>3x7x9',
    ),
    'outconv_reduce_kernel': (
        'outconv_bwd:bf16:1x16>2x12x9',
        'outconv_bwd:bf16:1x16>4x14x11',
        'outconv_bwd:bf16:1x16>6x16x13',
        'outconv_bwd:bf16:1x16>8x18x15',
        'outconv_bwd:bf16:1x6>3x7x9',
        'outconv_bwd:bf16:2x64>1x11x8',
        'outconv_bwd:bf16:2x64>3x13x10',
        'outconv_bwd:bf16:2x64>5x15x12',
        'outconv_bwd:bf16:2x64>7x17x14',
        'outconv_bwd:fp32:1x16>2x12x9',
        'outconv_bwd:fp32:1x16>4x14x11',
        'outconv_bwd:fp32:1x16>6x16x13',
        'outconv_bwd:fp32:1x16>8x18x15',
        'outconv_bwd:fp32:1x6>3x7x9',
        'outconv_bwd:fp32:2x64>1x11x8',
        'outconv_bwd:fp32:2x64>3x13x10',
        'outconv_bwd:fp32:2x64>5x15x12',
        'outconv_bwd:fp32:2x64>7x17x14',
        'outconv_bwd_bnbwd:bf16:1x16>2x12x9',
        'outconv_bwd_bnbwd:bf16:1x16>4x14x11',
        'outconv_bwd_bnbwd:bf16:1x16>6x16x13',
        'outconv_bwd_bnbwd:bf16:1x16>8x18x15',
        'outconv_bwd_bnbwd:bf16:2x64>1x11x8',
        'outconv_bwd_bnbwd:bf16:2x64>3x13x10',
        'outconv_bwd_bnbwd:bf16:2x64>5x15x12',
        'outconv_bwd_bnbwd:bf16:2x64>7x17x14',
        'outconv_bwd_bnbwd:fp32:1x16>2x12x9',
        'outconv_bwd_bnbwd:fp32:1x16>4x14x11',
        'outconv_bwd_bnbwd:fp32:1x16>6x16x13',
        'outconv_bwd_bnbwd:fp32:1x16>8x18x15',
        'outconv_bwd_bnbwd:fp32:2x64>1x11x8',
        'outconv_bwd_bnbwd:fp32:2x64>3x13x10',
        'outconv_bwd_bnbwd:fp32:2x64>5x15x12',
        'outconv_bwd_bnbwd:fp32:2x64>7x17x14',
    ),
}


def entry_kind(e):
    return e[0] if isinstance(e[0], str) and e[0] in ("env", "unreachable") else "cases"


def entry_cases(e):
    k = entry_kind(e)
    return () if k == "unreachable" else (e[2] if k == "env" else e)


_BY_CASE = {}
for _k, _e in LEDGER.items():
    for _c in entry_cases(_e):
        _BY_CASE.setdefault(_c, set()).add(_k)


def expected_kernels(cid):
    return _BY_CASE.get(cid, set())


# ------------------------------------------------------------------------------------------------
# running a set
# ------------------------------------------------------------------------------------------------
def run_set(name, strict=True):
    """run every case of switch set `name` in this process (its switches must already be in the environment).
    The cases name their own compute type: UNET_B200_PRECISION, which the fp32 wrappers read at each call
    (tf32x3 splits every fp32 tensor-core operand into three), is unset while they run, whatever an earlier user of
    the process left in it."""
    saved = os.environ.pop("UNET_B200_PRECISION", None)
    try:
        return _run_cases(name, strict)
    finally:
        if saved is not None:
            os.environ["UNET_B200_PRECISION"] = saved


def _run_cases(name, strict):
    res = {}
    for c in CASES:
        if c.env != name:
            continue
        try:
            r = run_case(c)
        except Exception as e:  # noqa: BLE001  (a case that cannot run is a failure of that case, reported with it)
            r = dict(kernels=[], worst=math.inf, rel=math.inf, failures=[f"{type(e).__name__}: {e}"])
        if strict:
            want = expected_kernels(c.id)
            if set(r["kernels"]) != want:
                extra, missing = sorted(set(r["kernels"]) - want), sorted(want - set(r["kernels"]))
                r["failures"].append(f"kernels differ from the ledger: launched but not listed {extra}, "
                                     f"listed but not launched {missing}")
        res[c.id] = r
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--set", default="default")
    ap.add_argument("--out", required=True)
    ap.add_argument("--no-strict", action="store_true")
    a = ap.parse_args()
    for k, v in ENV_SETS[a.set].items():
        assert os.environ.get(k) == v, f"switch {k} must be set in the environment of this process"
    res = run_set(a.set, strict=not a.no_strict)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
