"""torch.autograd.Function wrappers of the UNet parts over the C ABI.

One Function per reference part (SURVEY.md section 8a):
  DoubleConvFn  -- unet_parts.py:7-24   conv3x3+BN+ReLU twice (optionally also emits MaxPool2d(2) of its
                                        output, and can write its output into a caller-owned NHWC buffer:
                                        that is how the skip concat of unet_parts.py:95 costs no copy)
  MaxPoolFn     -- unet_parts.py:32     standalone MaxPool2d(2)
  UpCatConvTFn  -- unet_parts.py:72-95  ConvTranspose2d(k2,s2)+bias, F.pad placement, cat([x2, x1])
  UpCatBilinearFn -- unet_parts.py:69-95 bilinear x2 (align_corners=True), F.pad placement, cat
  OutConvFn     -- unet_parts.py:100-106 1x1 conv + bias
forward/backward only marshal pointers; all arithmetic happens in libunetb200.so.
"""
from __future__ import annotations

import os

import torch

from . import _lib, ops
from ._lib import ALGO_AUTO, ALGO_PREFER_TC, ALGO_SIMT


# ------------------------------------------------------------------------------------------------
# precision policy
# ------------------------------------------------------------------------------------------------
def compute_dtype(x):
    """bf16 whenever autocast is on (the reference's AMP path, train.py:116; evaluate.py:43;
    predict.py:22 -- BASELINE's bf16 mode) or the input already is bf16; fp32 otherwise."""
    if torch.is_autocast_enabled("cuda") or x.dtype == torch.bfloat16:
        return torch.bfloat16
    return torch.float32


def conv_algo(dtype):
    """bf16 -> tcgen05 when the layer shape fits.  fp32 -> UNET_B200_PRECISION: 'tf32' runs the
    tcgen05 kind::tf32 engine (what cuDNN does for the reference with allow_tf32=True), 'tf32x3' the
    same engine on hi/lo-split operands (three MMAs per product: fp32-level results, north_star's
    1e-3 mode on the tensor cores), 'fp32' exact fp32 FMAs on the CUDA cores."""
    if dtype == torch.bfloat16:
        return ALGO_AUTO
    mode = os.environ.get("UNET_B200_PRECISION", "").lower()
    if mode == "":
        mode = "tf32" if torch.backends.cudnn.allow_tf32 else "fp32"
    if mode in ("tf32", "tf32x3"):       # tf32x3: the 3-term split of ops.x3_active (fp32-level results)
        return ALGO_PREFER_TC
    if mode == "fp32":
        return ALGO_SIMT
    raise ValueError(f"UNET_B200_PRECISION must be 'tf32', 'tf32x3' or 'fp32', got {mode!r}")


def _w_src(w):
    """(fp32 tensor, s_out, s_in, s_tap) for a [O, I, kh, kw] parameter whose taps are linear in
    memory (contiguous or channels_last, cf. train.py:262 `.to(memory_format=channels_last)`)."""
    w = w.detach()
    if w.dtype != torch.float32:
        w = w.float()
    so, si, skh, skw = w.stride()
    kh, kw = w.shape[2], w.shape[3]
    if skh != kw * skw:          # taps must be linear in memory: t = kh*KW + kw -> t * skw
        w = w.contiguous()
        so, si, skh, skw = w.stride()
    return w, so, si, skw


def _job3x3_fprop(w):
    """OIHW -> Wp[co][(kh,kw)][ci]"""
    Co, Ci = w.shape[:2]
    w, so, si, st = _w_src(w)
    return w, (Co, 9, Ci), (so, st, si), 0, (Co, 9 * Ci)


def _job3x3_dgrad(w):
    """OIHW -> Wp[ci][(kh',kw')][co] = W[co][ci][2-kh'][2-kw']"""
    Co, Ci = w.shape[:2]
    w, so, si, st = _w_src(w)
    return w, (Ci, 9, Co), (si, -st, so), 8 * st, (Ci, 9 * Co)


def _jobT_fprop(w):
    """IOHW [Ci,Co,2,2] -> Wp[(q,co)][ci]"""
    Ci, Co = w.shape[:2]
    w, s_ci, s_co, st = _w_src(w)
    return w, (4, Co, Ci), (st, s_co, s_ci), 0, (4 * Co, Ci)


def _jobT_dgrad(w):
    """IOHW -> Wp[ci][(q,co)]"""
    Ci, Co = w.shape[:2]
    w, s_ci, s_co, st = _w_src(w)
    return w, (Ci, 4, Co), (s_ci, st, s_co), 0, (Ci, 4 * Co)


_JOBS = {"f3": _job3x3_fprop, "d3": _job3x3_dgrad, "fT": _jobT_fprop, "dT": _jobT_dgrad}


def _pack_many(items, dtype):
    """items: [(parameter, kind)] -> list of packed GEMM operands, written by ONE multi-tensor launch into one
    buffer (the weights of a network change together, at the optimizer step)."""
    specs = [_JOBS[kind](w) for w, kind in items]
    sizes = [sh[0] * sh[1] for _, _, _, _, sh in specs]
    starts, total = [], 0
    for n in sizes:
        starts.append(total)
        total += (n + 127) // 128 * 128            # keep every operand 256-byte aligned (TMA needs 16)
    flat = torch.empty(total, dtype=dtype, device=items[0][0].device)
    jobs = (_lib.PackJob * len(specs))()
    outs = []
    es = flat.element_size()
    for j, ((src, n, st, off, shape), o) in enumerate(zip(specs, starts)):
        jobs[j].src, jobs[j].dst = src.data_ptr(), flat.data_ptr() + o * es
        jobs[j].n0, jobs[j].n1, jobs[j].n2 = n
        jobs[j].s0, jobs[j].s1, jobs[j].s2 = st
        jobs[j].off = off
        outs.append(flat[o:o + shape[0] * shape[1]].view(shape))
    ops._run("pack_weights", ops.lib().unetb200_pack_weights_multi, jobs, len(specs), ops._DT[dtype], ops._stream(),
             nbytes=float(sum(sizes)) * (4 + es))
    return outs


# Replaying a captured CUDA graph moves weights and BatchNorm running statistics through raw pointers without
# touching any version counter.  Every replay advances this generation, and the caches below (packed operands,
# eval-mode BatchNorm coefficients) include it in their keys.
_GENERATION = [0]


def graph_replayed():
    """Mark every cached packed weight operand and eval-mode BatchNorm coefficient stale.  GraphedStep.replay and
    SegmentedStep.replay call it; call it after each replay of a graph captured with torch.cuda.graph directly."""
    _GENERATION[0] += 1


# GEMM operands packed ahead of their use by one launch at the start of a whole-network forward (`prepack`).  An
# entry is valid while the parameter object, its storage, its version counter, dtype, device and the replay
# generation are unchanged: FusedRMSprop bumps the version of every tensor it updates through raw pointers, so a
# cached operand can never outlive its weights (and inference re-uses the operands across calls: no pack launch at all).
_PRE = {}          # (id(w), kind) -> (packed, dtype, parameter version, weakref(w), data_ptr, generation)


def _pre_valid(ent, w, dtype):
    return (ent is not None and ent[1] == dtype and ent[2] == w._version and ent[3]() is w
            and ent[4] == w.data_ptr() and ent[0].device == w.device and ent[5] == _GENERATION[0])


def _packed(w, dtype, kind):
    ent = _PRE.get((id(w), kind))
    if _pre_valid(ent, w, dtype):
        return ent[0]
    return _pack_many([(w, kind)], dtype)[0]


def prepack(model, dtype, need_dgrad):
    """Pack every 3x3 / transposed conv weight of `model` into its fprop (and dgrad) GEMM operand: one launch."""
    import weakref
    jobs = []
    for m in model.modules():
        if isinstance(m, torch.nn.ConvTranspose2d) and m.kernel_size == (2, 2):
            jobs.append((m.weight, "fT"))
            if need_dgrad:
                jobs.append((m.weight, "dT"))
        elif isinstance(m, torch.nn.Conv2d) and m.kernel_size == (3, 3):
            jobs.append((m.weight, "f3"))
            if need_dgrad and m.in_channels >= 16:       # the first layer has no data gradient
                jobs.append((m.weight, "d3"))
    if not jobs or not all(w.is_cuda for w, _ in jobs):
        return False
    # a training step being captured into a CUDA graph must contain its own pack launch: on replay the weights have
    # moved although no Python-visible version counter has
    force = need_dgrad and torch.cuda.is_current_stream_capturing()
    todo = [(w, kind) for w, kind in jobs if force or not _pre_valid(_PRE.get((id(w), kind)), w, dtype)]
    if len(_PRE) > 4 * len(jobs) + 64:                  # entries of parameters that no longer exist
        for key in [k for k, e in _PRE.items() if e[3]() is None]:
            del _PRE[key]
    if todo:
        for (w, kind), packed in zip(todo, _pack_many(todo, dtype)):
            _PRE[(id(w), kind)] = (packed, dtype, w._version, weakref.ref(w), w.data_ptr(), _GENERATION[0])
    return True


def pack3x3_fprop(w, dtype):
    """OIHW -> Wp[co][(kh,kw)][ci]"""
    return _packed(w, dtype, "f3")


def pack3x3_dgrad(w, dtype):
    """OIHW -> Wp[ci][(kh',kw')][co] = W[co][ci][2-kh'][2-kw']"""
    return _packed(w, dtype, "d3")


def packT_fprop(w, dtype):
    """IOHW [Ci,Co,2,2] -> Wp[(q,co)][ci]"""
    return _packed(w, dtype, "fT")


def packT_dgrad(w, dtype):
    """IOHW -> Wp[ci][(q,co)]"""
    return _packed(w, dtype, "dT")


# ------------------------------------------------------------------------------------------------
# gradient sinks: where a parameter's gradient is to be written
# ------------------------------------------------------------------------------------------------
# A data-parallel reducer (ddp.GradAllReducer) registers, per parameter, an fp32 view of its all-reduce bucket
# with the parameter's shape and strides.  The backward kernels then write the gradient straight into the bucket
# (no per-step copy of 124 MB into the buckets); autograd receives a fresh alias of that view, so AccumulateGrad
# adopts it as p.grad without a copy.  Used only when nothing has to be accumulated: p.grad is None, or the
# reducer runs backward through torch.autograd.grad and owns p.grad (`always`).
_GRAD_SINK = {}    # id(param) -> (weakref(param), view, always)


def set_grad_sinks(params, views, always=False):
    import weakref
    for p, v in zip(params, views):
        if v.dtype != torch.float32 or v.shape != p.shape or v.stride() != p.stride():
            raise ValueError("unetb200: a gradient sink must be an fp32 tensor with the parameter's shape and strides")
        _GRAD_SINK[id(p)] = (weakref.ref(p), v, bool(always))


def clear_grad_sinks(params=None):
    if params is None:
        _GRAD_SINK.clear()
    else:
        for p in params:
            _GRAD_SINK.pop(id(p), None)


def grad_dst(param, like=None):
    """Fresh alias of `param`'s gradient sink if one is registered and usable now, else None."""
    ent = _GRAD_SINK.get(id(param))
    if ent is None or ent[0]() is not param:
        return None
    if not ent[2] and getattr(param, "grad", None) is not None:
        return None
    if like is not None and (tuple(like.shape) != tuple(ent[1].shape) or like.stride() != ent[1].stride()):
        return None
    return ent[1].detach()


# ------------------------------------------------------------------------------------------------
# BatchNorm-backward reductions made by the kernel that PRODUCES a gradient (cross-Function hand-off)
# ------------------------------------------------------------------------------------------------
# forward: a conv-BN-ReLU stage registers, for its activation z = relu(bn(y)), the pair (y, coefs) that its backward
# reduction needs; the consumer of z (OutConv, ...) looks it up and saves it.  backward: the consumer's kernel writes
# the gradient g of z and, in the same pass, sum(g*mask) / sum(g*mask*xhat); it leaves them here keyed by g's
# storage, and the stage's own backward takes them instead of running unetb200_bn_relu_bwd_reduce.
_BNBWD_MIN_N = int(os.environ.get("UNETB200_BNBWD_MIN_N", "0"))        # A/B switches: fuse only for these widths
_BNBWD_MAX_N = int(os.environ.get("UNETB200_BNBWD_MAX_N", "1000000"))
_BN_OF_ACT = {}    # data_ptr(z) -> (weakref(y), weakref(coefs), shape)
_GRAD_SUMS = {}    # data_ptr(g) -> (sums, shape)


# Column sums of a gradient made by the dgrad that writes it: the ConvTranspose2d bias gradient (unet_parts.py:73) is
# the per-channel sum of the `up` half of the concat gradient, which the decoder's first conv's dgrad produces -- its
# epilogue already knows how to sum the tile it stores (the forward BatchNorm statistics path).
# Both hand-offs carry a per-call token, so an entry that was never consumed can never be mistaken for another call's
# (addresses repeat once the allocator recycles a block).
_WANT_COLSUM = {}    # data_ptr(concat buffer) -> (shape, token): registered by UpCatConvTFn.forward, read by DoubleConvFn.forward
_GRAD_COLSUM = {}    # data_ptr(concat gradient) -> (fp64 stats[2*C], shape, token)
COLSUM_FUSE = os.environ.get("UNETB200_COLSUM_FUSE", "1") != "0"


def register_bn_of(z, y, coefs):
    import weakref
    if len(_BN_OF_ACT) > 256:
        for k in [k for k, e in _BN_OF_ACT.items() if e[0]() is None]:
            del _BN_OF_ACT[k]
    _BN_OF_ACT[z.data_ptr()] = (weakref.ref(y), weakref.ref(coefs), tuple(z.shape))


def bn_of(z):
    ent = _BN_OF_ACT.get(z.data_ptr())
    if ent is None or ent[2] != tuple(z.shape):
        return None
    y, coefs = ent[0](), ent[1]()
    if y is None or coefs is None or y.shape != z.shape or y.dtype != z.dtype:
        return None
    return y, coefs


def begin_forward():
    """Entry of a drop-in forward pass.  Outside any backward pass, whatever a backward pass left queued or handed
    off belongs to a pass that raised (train.py's OOM retry takes this route): drop it before it can reach the next
    pass.  Inside one (re-computation under use_checkpointing) nothing changes."""
    if _GRAD_SUMS or _GRAD_COLSUM:
        task = ops.graph_task()
        if task is not None and task < 0:
            _GRAD_SUMS.clear()
            _GRAD_COLSUM.clear()
    ops.drop_aborted_work_if_idle()


def leave_grad_sums(g, sums):
    if len(_GRAD_SUMS) > 64:
        _GRAD_SUMS.clear()
    _GRAD_SUMS[g.data_ptr()] = (sums, tuple(g.shape))


def take_grad_sums(g):
    ent = _GRAD_SUMS.pop(g.data_ptr(), None)
    if ent is None or ent[1] != tuple(g.shape):
        return None
    return ent[0]


def _f32c(t):
    t = t.detach()
    if t.dtype != torch.float32 or not t.is_contiguous():
        t = t.float().contiguous()
    return t


# ------------------------------------------------------------------------------------------------
# conv3x3 + BN + ReLU stage
# ------------------------------------------------------------------------------------------------
def _gconv3x3(x, Cout, y, dtype):
    B, Cin, H, W = x.shape
    return ops.make_gconv(ops._DT[dtype], conv_algo(dtype), B, H, W, Cin, ops.TAPS3, 1, (0, 0), H, W, ops.nhwc_ld(x),
                          Cout, 1, 1, (0, 0), H, W, ops.nhwc_ld(y))


# One zero-fill per forward pass for all the BatchNorm statistics accumulators of a network (18 tiny fills otherwise):
# the model opens an arena (`zero_arena`), conv_bn_relu_fwd takes fp64 slices from it; outside an arena, or when it is
# exhausted, a slice is an ordinary torch.zeros.
_ZERO_ARENA = [None, 0]


class zero_arena:
    def __init__(self, n_doubles, device):
        self.n, self.device = int(n_doubles), device

    def __enter__(self):
        self.prev = list(_ZERO_ARENA)
        _ZERO_ARENA[0] = torch.zeros(self.n, dtype=torch.float64, device=self.device) if self.n > 0 else None
        _ZERO_ARENA[1] = 0

    def __exit__(self, *exc):
        _ZERO_ARENA[0], _ZERO_ARENA[1] = self.prev
        return False


def zeros_f64(n, device):
    buf, off = _ZERO_ARENA
    n2 = (n + 1) // 2 * 2                      # keep slices 16-byte aligned
    if buf is not None and buf.device == torch.device(device) and off + n2 <= buf.numel() and not _RECOMPUTE[0]:
        _ZERO_ARENA[1] = off + n2
        return buf[off:off + n]
    return torch.zeros(n, dtype=torch.float64, device=device)


# Activation re-computation (UNet.use_checkpointing, reference unet_model.py:40-50 / train.py:294-299): while a
# checkpointed stage is re-run inside the backward pass its BatchNorm layers must normalise with the same batch
# statistics but leave the running statistics and num_batches_tracked alone (the first run already moved them).
_RECOMPUTE = [False]


class recompute_mode:
    """Context manager torch.utils.checkpoint enters around the re-run of a stage (context_fn)."""

    def __enter__(self):
        self.prev, _RECOMPUTE[0] = _RECOMPUTE[0], True

    def __exit__(self, *exc):
        _RECOMPUTE[0] = self.prev
        return False


# eval-mode BatchNorm coefficients (scale / shift from the running statistics), cached per module while the four
# tensors they come from are unchanged and no graph has been replayed since: an inference loop (evaluate.py:43-143, predict.py:22-27) then launches none
# of the 18 tiny coefficient kernels per forward
_EVAL_COEFS = {}    # id(bn) -> (weakref(bn), key, coefs)


def _eval_coefs(bn, Cout):
    import weakref
    parts = (bn.weight, bn.bias, bn.running_mean, bn.running_var)
    key = tuple((t.data_ptr(), t._version, t.dtype, t.device) if t is not None else None for t in parts) + (
        bn.eps, _GENERATION[0])
    ent = _EVAL_COEFS.get(id(bn))
    if ent is not None and ent[0]() is bn and ent[1] == key and not torch.cuda.is_current_stream_capturing():
        return ent[2]
    gamma = _f32c(bn.weight) if bn.weight is not None else None
    beta = _f32c(bn.bias) if bn.bias is not None else None
    coefs = ops.bn_eval_coeffs(gamma, beta, bn.running_mean, bn.running_var, bn.eps, Cout)
    if len(_EVAL_COEFS) > 512:
        for k in [k for k, e in _EVAL_COEFS.items() if e[0]() is None]:
            del _EVAL_COEFS[k]
    if not torch.cuda.is_current_stream_capturing():
        _EVAL_COEFS[id(bn)] = (weakref.ref(bn), key, coefs)
    return coefs


def sync_peer(bn, training, device):
    """The ddp.BNPeerGroup whose ranks a training-mode nn.SyncBatchNorm holder takes its statistics from, or None:
    BatchNorm2d holders, eval mode, and SyncBatchNorm without torch.distributed or in a group of one rank run the
    per-replica path unchanged (no extra launch)."""
    if not training or not isinstance(bn, torch.nn.SyncBatchNorm):
        return None
    from . import ddp
    return ddp.bn_sync_group(bn, device)


def conv_bn_relu_fwd(x, w, bn, training, out=None, want_pool=False, fold=False, outconv=None, peer=None):
    """x NHWC -> (y raw conv output, z = relu(bn(y)), pooled or None, coefs[4,C]).

    peer: the BNPeerGroup of a synchronised BatchNorm (sync_peer): the batch statistics are those of every rank.

    outconv = (weight [K, C, 1, 1], bias or None) with fold=True: when the fused kernel covers the shape, z is the
    LOGITS of OutConv applied to the activation ([B, K, H, W] view of a packed NHWC tensor) and the 5th return value
    is True; the activation itself is never written.

    fold=True (no backward will follow) with running statistics: BatchNorm + ReLU are folded into the conv epilogue
    (one write of z, no y; SURVEY section 8(f) N1) when the fused tcgen05 kernel covers the shape."""
    B, Cin, H, W = x.shape
    Cout = w.shape[0]
    cd, dev = x.dtype, x.device
    wp = pack3x3_fprop(w, cd)
    if fold and not (training or bn.running_mean is None) and Cout % 2 == 0:
        if outconv is not None and out is None and not want_pool:
            ow, ob = outconv
            K = ow.shape[0]
            d = ops.make_gconv(ops._DT[cd], conv_algo(cd), B, H, W, Cin, ops.TAPS3, 1, (0, 0), H, W, ops.nhwc_ld(x),
                               Cout, 1, 1, (0, 0), H, W, Cout)
            if tuple(ow.shape[1:]) == (Cout, 1, 1) and ops.gconv_fprop_affine_relu_outconv_supported(d, x, wp, K):
                coefs = _eval_coefs(bn, Cout)
                logits = torch.empty((B, H, W, K), dtype=cd, device=dev)
                ops.gconv_fprop_affine_relu_outconv(d, x, wp, coefs, _f32c(ow).view(K, Cout),
                                                    _f32c(ob) if ob is not None else None, logits)
                return None, logits.permute(0, 3, 1, 2), None, coefs, True
        z = out if out is not None else ops.empty_nhwc(B, Cout, H, W, cd, dev)
        d = _gconv3x3(x, Cout, z, cd)
        if ops.gconv_fprop_affine_relu_supported(d, x, wp, z):
            coefs = _eval_coefs(bn, Cout)
            pooled = ops.empty_nhwc(B, Cout, H // 2, W // 2, cd, dev) if want_pool else None
            if pooled is not None and ops.gconv_fprop_affine_relu_pool_supported(d, x, wp, z, pooled):
                ops.gconv_fprop_affine_relu(d, x, wp, coefs, z, pooled)      # the pool rides in the conv epilogue
            else:
                ops.gconv_fprop_affine_relu(d, x, wp, coefs, z)
                if pooled is not None:
                    ops.maxpool2_fwd(z, pooled)
            return None, z, pooled, coefs, False
    y = ops.empty_nhwc(B, Cout, H, W, cd, dev)
    use_batch = training or bn.running_mean is None
    stats = zeros_f64(2 * Cout, dev) if use_batch else None
    ops.gconv_fprop(_gconv3x3(x, Cout, y, cd), x, wp, None, y, stats)
    gamma = _f32c(bn.weight) if bn.weight is not None else None
    beta = _f32c(bn.bias) if bn.bias is not None else None
    if use_batch:
        if bn.momentum is None and bn.running_mean is not None and training:
            raise ValueError(f"unetb200: {type(bn).__name__}(momentum=None) (cumulative average) is not supported")
        update = training and bn.running_mean is not None and not _RECOMPUTE[0]
        args = (stats, B * H * W, gamma, beta, bn.eps, bn.momentum if update else 0.0,
                bn.running_mean if update else None, bn.running_var if update else None, Cout)
        nbt = bn.num_batches_tracked if update else None
        if peer is None:
            coefs = ops.bn_finalize(*args, num_batches_tracked=nbt)
        else:
            coefs = ops.bn_sync_finalize(peer, *args, num_batches_tracked=nbt)
        if update:
            # the kernel moved the running statistics through raw pointers: tell PyTorch (autograd's saved-tensor
            # check, the eval-coefficient cache above)
            torch._C._increment_version([bn.running_mean, bn.running_var])
    else:
        coefs = ops.bn_eval_coeffs(gamma, beta, bn.running_mean, bn.running_var, bn.eps, Cout)
    z = out if out is not None else ops.empty_nhwc(B, Cout, H, W, cd, dev)
    pooled = ops.empty_nhwc(B, Cout, H // 2, W // 2, cd, dev) if want_pool else None
    ops.bn_relu_apply(y, coefs, z, pooled)
    return y, z, pooled, coefs, False


def _grad_kept_as_is(param, dW):
    """True when autograd will simply keep `dW` as `param.grad` without reading it on the current stream: no
    existing .grad to accumulate into, same layout and dtype (AccumulateGrad's layout contract), no tensor hooks
    that would look at the gradient during backward, and not a double-backward pass.  Only then may the weight
    gradient be produced on the side stream."""
    if getattr(param, "grad", None) is not None or torch.is_grad_enabled():
        return False
    if dW.stride() != param.stride() or param.dtype != torch.float32 or dW.dtype != torch.float32:
        return False
    if getattr(param, "_backward_hooks", None) or getattr(param, "_post_accumulate_grad_hooks", None):
        return False
    return True


def _sink_owns(param, dW):
    """True when dW IS the registered gradient sink of `param` in `always` mode: the data-parallel reducer drives the
    backward pass through torch.autograd.grad and owns p.grad, so nothing reads dW before the pass (segment) ends."""
    ent = _GRAD_SINK.get(id(param))
    return (ent is not None and ent[0]() is param and ent[2] and dW.data_ptr() == ent[1].data_ptr()
            and not torch.is_grad_enabled())


def _defer_mode(param, dW, kept, side):
    """gconv_wgrad's `defer` for the weight gradient dW of `param`: "pass" when a data-parallel sink owns it (its split
    reduction joins the one launch at the end of the backward pass); "call" when autograd keeps dW as it is (one
    launch for the layers of the running Function's backward, before autograd sees dW); else, and on the side stream,
    the reduction follows its wgrad.  Deferred reductions all run on the multi-tensor kernel, whose per-layer
    summation order does not depend on how the layers are grouped."""
    if side:
        return False
    if _sink_owns(param, dW):
        return "pass"
    return "call" if kept else False


def _vec_dst(param, Cc):
    """gradient sink of a [C] parameter (BatchNorm gamma / beta, a bias), if any"""
    if param is None:
        return None
    d = grad_dst(param)
    return d if d is not None and d.dim() == 1 and d.numel() == Cc and d.is_contiguous() else None


def conv_bn_relu_bwd(gz, x, y, w, coefs, batch_stats, need_gx, param=None, bn_params=(None, None), sums=None,
                     below=None, colsum=None, peer=None):
    """-> (gx or None, dW [Co,Ci,3,3] fp32, dgamma, dbeta, sums_below).  `param`: the Parameter object behind `w`;
    `bn_params`: the BatchNorm weight / bias Parameter objects (only to look up their gradient sinks); `sums`: the
    BatchNorm-backward reduction of THIS stage if the kernel that produced gz already made it; `below` = (y, coefs)
    of the conv-BN-ReLU stage whose activation is `x`: its reduction is then made by this stage's dgrad epilogue
    when the fused kernel covers the shape and returned as sums_below (else None).  `peer`: as conv_bn_relu_fwd."""
    param = w if param is None else param
    B, Cin, H, W = x.shape
    Cout = w.shape[0]
    cd = x.dtype
    gy, dgamma, dbeta = ops.bn_relu_bwd(gz, y, coefs, batch_stats, _vec_dst(bn_params[0], Cout),
                                        _vec_dst(bn_params[1], Cout), sums=sums, peer=peer)
    # the gradient takes the parameter's own memory layout (OIHW or channels_last): AccumulateGrad then keeps it
    # without a copy, and for channels_last the split reduction writes it coalesced; with a registered sink
    # (data-parallel bucket view) it is written there
    dW = grad_dst(param)
    if dW is None:
        dW = torch.empty_like(w, dtype=torch.float32)
    so, si, skh, skw = dW.stride()
    if skh != 3 * skw or dW.shape != (Cout, Cin, 3, 3):
        dW = torch.empty((Cout, Cin, 3, 3), dtype=torch.float32, device=x.device)
        so, si, skh, skw = dW.stride()
    gx = None
    dw_desc = _gconv3x3(x, Cout, gy, cd)
    gs = ops.x3_split(gy) if (ops.x3_active(dw_desc) and Cout >= 16) else None   # 3xTF32: one split serves both GEMMs
    sums_below = None
    if need_gx:
        gx = ops.empty_nhwc(B, Cin, H, W, cd, x.device)
        dd = _gconv3x3(gy, Cin, gx, cd)
        wd = pack3x3_dgrad(w, cd)
        if (below is not None and gs is None and _BNBWD_MIN_N <= Cin <= _BNBWD_MAX_N
                and ops.gconv_dgrad_bnbwd_supported(dd, gy, wd, gx)):
            sums_below = ops.gconv_dgrad_bnbwd(dd, gy, wd, gx, below[0], below[1])
        elif colsum is not None and colsum is not False and gs is None:
            # x is an Up stage's concat buffer: leave the per-channel sums of its gradient for the ConvTranspose bias
            cs = torch.zeros(2 * Cin, dtype=torch.float64, device=x.device)
            ops.gconv_fprop(dd, gy, wd, None, gx, cs, kind="dgrad")
            if len(_GRAD_COLSUM) > 16:
                _GRAD_COLSUM.clear()
            _GRAD_COLSUM[gx.data_ptr()] = (cs, tuple(gx.shape), colsum)
        else:
            ops.gconv_fprop(dd, gy, wd, None, gx, None, kind="dgrad", x_split=gs)
    # after the dgrad, on the side stream: overlaps the (memory-bound) BatchNorm backward of the previous layer
    # (only when AccumulateGrad will simply keep dW: an existing .grad would be accumulated into on the main stream)
    kept = _grad_kept_as_is(param, dW)
    side = kept and ops.wgrad_on_side_stream()
    defer = _defer_mode(param, dW, kept, side)
    run = lambda: ops.gconv_wgrad(dw_desc, x, gy, dW, skw, si, so, gy_split=gs, defer=defer)  # noqa: E731
    if side:
        ops.on_side_stream(run, x, gy)      # AccumulateGrad keeps dW as it is (same layout, no other owner)
    else:
        run()                               # (else it would accumulate / re-layout dW on the main stream right away)
    return gx, dW, dgamma, dbeta, sums_below


class ToNHWCFn(torch.autograd.Function):
    """Layout / dtype conversion of a caller tensor into the internal NHWC form (a strided gather)."""

    @staticmethod
    def forward(ctx, x, dtype):
        ctx.in_dtype = x.dtype
        return ops.to_nhwc(x, dtype)

    @staticmethod
    def backward(ctx, g):
        dt = ctx.in_dtype if ctx.in_dtype in ops._DT else torch.float32
        return ops.to_nhwc(g, dt), None


class CutFn(torch.autograd.Function):
    """Identity that gives a tensor its own autograd node: a cut point of a segmented backward pass
    (unetb200.ddp.segmented_backward).  torch.autograd.grad(..., inputs=[t]) executes every node from which t's
    PRODUCER can be reached -- for a skip tensor that is the whole rest of the network (its producer also emits the
    pooled tensor the deeper stages consume).  Requesting the gradient at the cut alias instead stops the engine
    there; the next segment then starts from the producer's own output with that gradient."""

    @staticmethod
    def forward(ctx, x):
        return x.view_as(x)

    @staticmethod
    def backward(ctx, g):
        return g


class _Cfg:
    """Non-tensor arguments of a Function call."""

    def __init__(self, **kw):
        self.__dict__.update(kw)


class DoubleConvFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, w1, g1, b1, w2, g2, b2, cfg):
        fold = not cfg.save
        ctx.peers = (sync_peer(cfg.bn1, cfg.training, x.device), sync_peer(cfg.bn2, cfg.training, x.device))
        y1, z1, _, c1, _ = conv_bn_relu_fwd(x, w1, cfg.bn1, cfg.training, fold=fold, peer=ctx.peers[0])
        y2, z2, pooled, c2, fused_out = conv_bn_relu_fwd(z1, w2, cfg.bn2, cfg.training, out=cfg.out,
                                                         want_pool=cfg.want_pool, fold=fold,
                                                         outconv=getattr(cfg, "outconv", None) if fold else None,
                                                         peer=ctx.peers[1])
        cfg.fused_outconv = fused_out          # tells the caller whether z2 already holds OutConv's logits
        ctx.batch_stats = (cfg.training or cfg.bn1.running_mean is None, cfg.training or cfg.bn2.running_mean is None)
        ctx.has_pool = pooled is not None
        want = _WANT_COLSUM.pop(x.data_ptr(), None) if cfg.save else None
        ctx.colsum = want[1] if (want is not None and want[0] == tuple(x.shape)) else None      # the Up stage's token
        if cfg.save:
            ctx.save_for_backward(x, y1, z1, y2, z2, c1, c2, w1, w2)
            ctx.param_objs = (w1, g1, b1, w2, g2, b2)   # the Parameter objects themselves (.grad / gradient sinks)
            if y2 is not None:
                register_bn_of(z2, y2, c2)
        if pooled is None:
            return z2
        return z2, pooled

    @staticmethod
    def backward(ctx, gz2, gpooled=None):
        with ops.reductions_at_return():          # both weight gradients complete before autograd sees them
            return DoubleConvFn._backward(ctx, gz2, gpooled)

    @staticmethod
    def _backward(ctx, gz2, gpooled):
        x, y1, z1, y2, z2, c1, c2, w1, w2 = ctx.saved_tensors
        cd = x.dtype
        gz = ops.to_nhwc(gz2, cd) if gz2 is not None else None
        # reduction of bn2's backward already made by the kernel that wrote gz (OutConv backward)?  Only valid while
        # gz is exactly that tensor: not after the pool gradient has been accumulated into it below.
        sums2 = take_grad_sums(gz) if gz is not None else None
        if ctx.has_pool and gpooled is not None:
            sums2 = None
            gp = ops.to_nhwc(gpooled, cd)
            if gz is None:
                gz = ops.empty_nhwc(*z2.shape, cd, x.device)
                ops.maxpool2_bwd(z2, gp, gz, accumulate=False)
            elif gz is gz2 and ops.nhwc_ld(gz) > gz.shape[1] and not os.environ.get("UNETB200_NO_INPLACE_SKIP"):
                # gz2 is the skip half of a concat-gradient buffer produced by our own dgrad: the
                # pool gradient is accumulated into it in place (skip-gradient sum fused away), and the same pass
                # makes the reduction of bn2's backward (gz is complete exactly here)
                if ops.POOL_BNBWD_FUSE and y2 is not None:
                    sums2 = ops.maxpool2_bwd_bnreduce(z2, gp, gz, y2, c2)
                else:
                    ops.maxpool2_bwd(z2, gp, gz, accumulate=True)
            else:
                t = ops.empty_nhwc(*z2.shape, cd, x.device)
                ops.maxpool2_bwd(z2, gp, t, accumulate=False)
                gz = ops.add_channels_(t, gz)
        if gz is None:
            raise RuntimeError("DoubleConvFn.backward called without any output gradient")
        need = ctx.needs_input_grad
        p1, pg1, pb1, p2, pg2, pb2 = getattr(ctx, "param_objs", (w1, None, None, w2, None, None))
        # conv2's dgrad output is the gradient of z1 = relu(bn1(y1)): its epilogue makes bn1's backward reduction
        gz1, dW2, dg2, db2, sums1 = conv_bn_relu_bwd(gz, z1, y2, w2, c2, ctx.batch_stats[1], True, param=p2,
                                                     bn_params=(pg2, pb2), below=(y1, c1), sums=sums2,
                                                     peer=ctx.peers[1])
        gx, dW1, dg1, db1, _ = conv_bn_relu_bwd(gz1, x, y1, w1, c1, ctx.batch_stats[0], need[0], param=p1,
                                                bn_params=(pg1, pb1), sums=sums1, colsum=ctx.colsum, peer=ctx.peers[0])
        return (gx, dW1 if need[1] else None, dg1 if need[2] else None, db1 if need[3] else None,
                dW2 if need[4] else None, dg2 if need[5] else None, db2 if need[6] else None, None)


class MaxPoolFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x):
        B, Cc, H, W = x.shape
        p = ops.empty_nhwc(B, Cc, H // 2, W // 2, x.dtype, x.device)
        ops.maxpool2_fwd(x, p)
        ctx.save_for_backward(x)
        return p

    @staticmethod
    def backward(ctx, gp):
        (x,) = ctx.saved_tensors
        gx = ops.empty_nhwc(*x.shape, x.dtype, x.device)
        ops.maxpool2_bwd(x, ops.to_nhwc(gp, x.dtype), gx, accumulate=False)
        return gx


# ------------------------------------------------------------------------------------------------
# Up: upsample + pad + concat
# ------------------------------------------------------------------------------------------------
def _cat_buffer(x2, Cup, cat):
    """NHWC [B, C2+Cup, H, W] buffer whose first C2 channels hold x2 (copied unless x2 already
    lives there, which is the case when UNet.forward pre-allocated the buffer)."""
    B, C2, H, W = x2.shape
    if cat is not None and cat.data_ptr() == x2.data_ptr() and ops.nhwc_ld(cat) == ops.nhwc_ld(x2) \
            and cat.shape == (B, C2 + Cup, H, W):
        return cat
    cat = ops.empty_nhwc(B, C2 + Cup, H, W, x2.dtype, x2.device)
    ops.copy_channels(x2, ops.channel_slice(cat, 0, C2))
    return cat


def _pad_offsets(x1, x2):
    dy = x2.shape[2] - 2 * x1.shape[2]
    dx = x2.shape[3] - 2 * x1.shape[3]
    if dy < 0 or dx < 0:
        raise ValueError("unetb200.Up: the upsampled tensor is larger than the skip tensor (negative F.pad / "
                         f"cropping, unet_parts.py:85-88) is not supported: x1 {tuple(x1.shape)}, x2 {tuple(x2.shape)}")
    return dy, dx, (dy // 2, dx // 2)


class UpCatConvTFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x1, x2, wT, bT, cfg):
        B, C1, h, w = x1.shape
        Cup = wT.shape[1]
        C2, H, W = x2.shape[1:]
        cd = x1.dtype
        dy, dx, off = _pad_offsets(x1, x2)
        cat = _cat_buffer(x2, Cup, cfg.cat)
        up = ops.channel_slice(cat, C2, Cup)
        if dy or dx:
            ops.zero_channels(up)
        d = ops.make_gconv(ops._DT[cd], conv_algo(cd), B, h, w, C1, ops.TAPS1, 1, (0, 0), h, w, ops.nhwc_ld(x1),
                           4 * Cup, 4, 2, off, H, W, ops.nhwc_ld(cat))
        ops.gconv_fprop(d, x1, packT_fprop(wT, cd), _f32c(bT) if bT is not None else None, up, None,
                        kind="convT_fprop")
        ctx.geom = (C2, Cup, off, dy or dx)
        if cfg.save:
            ctx.save_for_backward(x1, wT)
            ctx.param_obj = wT
            ctx.bias_obj = bT
            if bT is not None and not (dy or dx) and COLSUM_FUSE:
                if len(_WANT_COLSUM) > 16:
                    _WANT_COLSUM.clear()
                ctx.colsum_token = object()
                _WANT_COLSUM[cat.data_ptr()] = (tuple(cat.shape), ctx.colsum_token)
        return cat

    @staticmethod
    def backward(ctx, gcat):
        with ops.reductions_at_return():          # the weight gradient is complete before autograd sees it
            return UpCatConvTFn._backward(ctx, gcat)

    @staticmethod
    def _backward(ctx, gcat):
        x1, wT = ctx.saved_tensors
        C2, Cup, off, padded = ctx.geom
        B, C1, h, w = x1.shape
        cd = x1.dtype
        g = ops.to_nhwc(gcat, cd)
        H, W = g.shape[2:]
        need = ctx.needs_input_grad
        g2 = ops.channel_slice(g, 0, C2) if need[1] else None
        gup = ops.channel_slice(g, C2, Cup)
        ld = ops.nhwc_ld(g)
        dW = dB = gx1 = None
        if need[2]:
            d = ops.make_gconv(ops._DT[cd], conv_algo(cd), B, h, w, C1, ops.TAPS1, 1, (0, 0), h, w, ops.nhwc_ld(x1),
                               4 * Cup, 4, 2, off, H, W, ld)
            # gradient in the parameter's own layout (see conv_bn_relu_bwd); quadrant q = kh*2 + kw must stay linear
            pT = getattr(ctx, "param_obj", wT)
            dW = grad_dst(pT)
            if dW is None:
                dW = torch.empty_like(wT, dtype=torch.float32)
            if dW.shape != (C1, Cup, 2, 2) or dW.stride(2) != 2 * dW.stride(3):
                dW = torch.empty((C1, Cup, 2, 2), dtype=torch.float32, device=g.device)
            s_ci, s_co, _, s_q = dW.stride()
        if need[0]:
            gx1 = ops.empty_nhwc(B, C1, h, w, cd, g.device)
            dd = ops.make_gconv(ops._DT[cd], conv_algo(cd), B, h, w, Cup, ops.TAPS_Q, 2, off, H, W, ld,
                                C1, 1, 1, (0, 0), h, w, ops.nhwc_ld(gx1))
            ops.gconv_fprop(dd, gup, packT_dgrad(wT, cd), None, gx1, None, kind="convT_dgrad")
        if need[2]:
            # after the dgrad, on the side stream (see conv_bn_relu_bwd)
            pT = getattr(ctx, "param_obj", wT)
            kept = _grad_kept_as_is(pT, dW)
            side = kept and ops.wgrad_on_side_stream()
            defer = _defer_mode(pT, dW, kept, side)
            run = lambda: ops.gconv_wgrad(d, x1, gup, dW, 0, s_ci, s_co, sq=s_q, defer=defer)  # noqa: E731
            if side:
                ops.on_side_stream(run, x1, g)
            else:
                run()
        cs = _GRAD_COLSUM.pop(g.data_ptr(), None)
        if need[3]:
            dst = _vec_dst(getattr(ctx, "bias_obj", None), Cup)
            if (cs is not None and cs[1] == tuple(g.shape) and cs[2] is getattr(ctx, "colsum_token", None)
                    and not padded and g is gcat):
                dB = ops.f64_to_f32(cs[0][C2:C2 + Cup], dst)      # summed by the dgrad epilogue that wrote g
            else:
                region = gup if not padded else ops.to_nhwc(
                    gup[:, :, off[0]:off[0] + 2 * h, off[1]:off[1] + 2 * w].contiguous(memory_format=torch.channels_last), cd)
                dB = ops.channel_sum(region, dst)
        return gx1, g2, dW, dB, None


class UpCatBilinearFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x1, x2, cfg):
        B, C1, h, w = x1.shape
        C2 = x2.shape[1]
        dy, dx, off = _pad_offsets(x1, x2)
        cat = _cat_buffer(x2, C1, cfg.cat)
        up = ops.channel_slice(cat, C2, C1)
        if dy or dx:
            ops.zero_channels(up)
        ops.upsample2x_fwd(x1, up, off)
        ctx.geom = (C2, C1, off, (B, C1, h, w), x1.dtype)
        return cat

    @staticmethod
    def backward(ctx, gcat):
        C2, C1, off, shape, cd = ctx.geom
        g = ops.to_nhwc(gcat, cd)
        need = ctx.needs_input_grad
        g2 = ops.channel_slice(g, 0, C2) if need[1] else None
        gx1 = None
        if need[0]:
            gx1 = ops.empty_nhwc(*shape, g.dtype, g.device)
            ops.upsample2x_bwd(ops.channel_slice(g, C2, C1), gx1, off)
        return gx1, g2, None


# ------------------------------------------------------------------------------------------------
# SpatialAttention gate (UNet_SA: unet_parts.py:39-60, applied to the skip tensor at :91-92)
# ------------------------------------------------------------------------------------------------
class SpatialGateFn(torch.autograd.Function):
    """x2 * sigmoid(conv7x7([mean_c x2, max_c x2])), written into ``cfg.out`` (the skip half of the concat buffer)."""

    @staticmethod
    def forward(ctx, x, w, cfg):
        B, Cc, H, W = x.shape
        if tuple(w.shape) != (1, 2, 7, 7):
            raise ValueError(f"unetb200: SpatialAttention supports the 7x7 kernel the reference builds, got {tuple(w.shape)}")
        out = cfg.out if cfg.out is not None else ops.empty_nhwc(B, Cc, H, W, x.dtype, x.device)
        wc = _f32c(w).reshape(-1)
        stats, gate = ops.sa_forward(x, wc, out)
        if cfg.save:
            ctx.save_for_backward(x, wc, stats, gate)
            ctx.param_obj = w
        return out

    @staticmethod
    def backward(ctx, gout):
        x, wc, stats, gate = ctx.saved_tensors
        g = ops.to_nhwc(gout, x.dtype)
        dx = ops.empty_nhwc(*x.shape, x.dtype, x.device)
        # the kernel writes dw as 98 contiguous values: into the gradient sink when that is laid out so
        dw = grad_dst(ctx.param_obj)
        if dw is None or not dw.is_contiguous():
            dw = torch.empty((1, 2, 7, 7), dtype=torch.float32, device=x.device)
        ops.sa_backward(g, x, wc, stats, gate, dx, dw)
        need = ctx.needs_input_grad
        return (dx if need[0] else None), (dw if need[1] else None), None


# ------------------------------------------------------------------------------------------------
# OutConv
# ------------------------------------------------------------------------------------------------
class OutConvFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, w, b, cfg):
        B, Cc, H, W = x.shape
        K = w.shape[0]
        logits = torch.empty((B, H, W, K), dtype=x.dtype, device=x.device)
        w2 = _f32c(w).view(K, Cc)
        ops.outconv_fwd(x, w2, _f32c(b) if b is not None else None, logits)
        ctx.below = False
        if cfg.save:
            below = bn_of(x)
            if below is not None:
                ctx.save_for_backward(x, w2, below[0], below[1])
                ctx.below = True
            else:
                ctx.save_for_backward(x, w2)
            ctx.param_objs = (w, b)
        ctx.has_bias = b is not None
        return logits.permute(0, 3, 1, 2)

    @staticmethod
    def backward(ctx, glogits):
        below = None
        if ctx.below:
            x, w2, yb, cb = ctx.saved_tensors
            below = (yb, cb)
        else:
            x, w2 = ctx.saved_tensors
        B, Cc, H, W = x.shape
        K = w2.shape[0]
        g = ops.to_nhwc(glogits, x.dtype, packed=True)
        need = ctx.needs_input_grad
        gx = ops.empty_nhwc(B, Cc, H, W, x.dtype, x.device) if need[0] else None
        pw, pb = getattr(ctx, "param_objs", (None, None))
        dw = grad_dst(pw) if pw is not None else None
        if dw is None or not dw.is_contiguous() and not dw.is_contiguous(memory_format=torch.channels_last):
            dw = torch.empty((K, Cc, 1, 1), dtype=torch.float32, device=x.device)
        db = _vec_dst(pb, K)
        if db is None:
            db = torch.empty(K, dtype=torch.float32, device=x.device)
        sums = ops.outconv_bwd(x, w2, g, gx, dw, db, below=below)
        if sums is not None:
            leave_grad_sums(gx, sums)      # x = relu(bn(yb)): the stage below takes them in its backward
        return gx, dw if need[1] else None, db if (need[2] and ctx.has_bias) else None, None
