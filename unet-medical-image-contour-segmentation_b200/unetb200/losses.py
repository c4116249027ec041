"""Loss-side autograd Functions over the C ABI.

  dice_coeff / multiclass_dice_coeff / dice_loss  -- reference utils/dice_score.py:5-36
  boundary_loss                                   -- reference utils/boundary_loss.py:5-118
  ce_dice_loss                                    -- the fused form of train.py:137-142
                                                     (CrossEntropyLoss + multiclass dice on softmax/one-hot)
  bce_dice_loss                                   -- the fused form of train.py:118-134 without its boundary term
                                                     (BCEWithLogitsLoss + dice on sigmoid, n_classes == 1)
  training_criterion                              -- either branch plus its boundary term
"""
from __future__ import annotations

import ctypes as C

import torch

from . import _lib, ops
from ._lib import BF16, F32, I64, U8


# ------------------------------------------------------------------------------------------------
# dice
# ------------------------------------------------------------------------------------------------
def _dense_same_layout(a, b):
    def dense(t):
        return t.is_contiguous() or (t.dim() == 4 and t.is_contiguous(memory_format=torch.channels_last))
    return (a.stride() == b.stride() and a.dtype == torch.float32 and b.dtype == torch.float32 and
            dense(a) and dense(b))


class DiceCoeffFn(torch.autograd.Function):
    """mean over G groups of (2*sum(x*t)+eps)/(sum x + sum t + eps), sets==0 -> inter (dice_score.py:14-18)."""

    @staticmethod
    def forward(ctx, x, t, G, eps):
        L = x.numel() // G
        dev = x.device
        acc = torch.empty(3 * G, dtype=torch.float64, device=dev)
        out = torch.empty(1, dtype=torch.float32, device=dev)
        saved = torch.empty(2 * G, dtype=torch.float32, device=dev)
        ops._run("dice_fwd", ops.lib().unetb200_dice_fwd, ops._p(x), ops._p(t), G, L, eps, ops._p(acc), ops._p(out),
                 ops._p(saved), ops._stream(), kernels=2, nbytes=8.0 * x.numel())
        ctx.save_for_backward(x, t, saved)
        ctx.G, ctx.eps = G, eps
        return out.reshape(())

    @staticmethod
    def backward(ctx, g):
        x, t, saved = ctx.saved_tensors
        G = ctx.G
        gs = g.detach().float().reshape(1).contiguous()
        gx = torch.empty_like(x)
        ops._run("dice_bwd", ops.lib().unetb200_dice_bwd, ops._p(x), ops._p(t), G, x.numel() // G, ctx.eps,
                 ops._p(saved), ops._p(gs), ops._p(gx), ops._stream(), nbytes=8.0 * x.numel())
        return gx, None, None, None


def dice_coeff(input, target, reduce_batch_first=False, epsilon=1e-6):
    assert input.size() == target.size()
    assert input.dim() == 3 or not reduce_batch_first
    ops.require_cuda(input, "dice_coeff")
    if input.dim() < 2:
        raise ValueError("dice_coeff expects at least 2-D inputs")
    if input.dim() == 2 or not reduce_batch_first:
        G = 1
        for s in input.shape[:-2]:
            G *= s
    else:
        G = 1
    x, t = input, target
    if not (G == 1 and _dense_same_layout(x, t)):
        # group-major contiguous fp32 (layout plumbing only)
        x = x.float().contiguous()
        t = t.float().contiguous()
    if x.numel() == 0:
        raise ValueError("dice_coeff: empty input")
    return DiceCoeffFn.apply(x, t, G, float(epsilon))


def multiclass_dice_coeff(input, target, reduce_batch_first=False, epsilon=1e-6):
    # reference: dice_coeff(input.flatten(0, 1), target.flatten(0, 1), ...)  (dice_score.py:30)
    if reduce_batch_first:
        # one global ratio over B*C*H*W: element order is irrelevant, no flatten copy needed
        assert input.size() == target.size()
        ops.require_cuda(input, "multiclass_dice_coeff")
        x, t = input, target
        if not _dense_same_layout(x, t):
            x = x.float().contiguous()
            t = t.float().contiguous()
        return DiceCoeffFn.apply(x, t, 1, float(epsilon))
    return dice_coeff(input.flatten(0, 1), target.flatten(0, 1), reduce_batch_first, epsilon)


def dice_loss(input, target, multiclass=False):
    fn = multiclass_dice_coeff if multiclass else dice_coeff
    return 1 - fn(input, target, reduce_batch_first=True)


# ------------------------------------------------------------------------------------------------
# boundary loss (value only: the reference's result has requires_grad=False by construction)
# ------------------------------------------------------------------------------------------------
@torch.no_grad()
def boundary_loss(pred_mask, target_mask, edge_width=64, edge_weight=5.0, smooth=1e-6):
    ops.require_cuda(pred_mask, "boundary_loss")
    pred = pred_mask.detach()
    if pred.dim() == 4:
        pred = pred[:, 1, :, :] if pred.size(1) > 1 else pred.squeeze(1)
    if pred.dim() != 3:
        raise ValueError(f"boundary_loss: pred_mask must be [B,H,W] or [B,C,H,W], got {tuple(pred_mask.shape)}")
    if pred.dtype not in (torch.float32, torch.bfloat16):
        pred = pred.float()
    tgt = target_mask.detach()
    if tgt.dtype == torch.float32:
        tdt = F32
    elif tgt.dtype == torch.int64:
        tdt = I64
    else:
        tgt = tgt.float()
        tdt = F32
    B, H, W = pred.shape
    if tuple(tgt.shape) != (B, H, W):
        raise ValueError(f"boundary_loss: target {tuple(tgt.shape)} does not match prediction {(B, H, W)}")
    if int(edge_width) != edge_width or edge_width < 0:
        raise ValueError("boundary_loss: edge_width must be a non-negative integer")
    L = ops.lib()
    work = torch.empty(L.unetb200_boundary_work_bytes(), dtype=torch.uint8, device=pred.device)
    out = torch.empty(1, dtype=torch.float32, device=pred.device)
    ops._run("boundary_loss", L.unetb200_boundary_loss, ops._p(pred), BF16 if pred.dtype == torch.bfloat16 else F32,
             *pred.stride(), ops._p(tgt), tdt, *tgt.stride(), B, H, W, int(edge_width), float(edge_weight),
             float(smooth), ops._p(work), ops._p(out), ops._stream(), kernels=2,
             nbytes=float(B * H * W) * (pred.element_size() + tgt.element_size()))
    return out.reshape(())


# ------------------------------------------------------------------------------------------------
# fused CE + dice criterion
# ------------------------------------------------------------------------------------------------
class CeDiceFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, logits, target, eps):
        B, K, H, W = logits.shape
        dev = logits.device
        acc = torch.empty(4, dtype=torch.float64, device=dev)
        out = torch.empty(4, dtype=torch.float32, device=dev)
        coefs = torch.empty(4, dtype=torch.float32, device=dev)
        ops._run("ce_dice_fwd", ops.lib().unetb200_ce_dice_fwd, ops._p(logits), ops.dt(logits), ops._p(target),
                 B * H * W, K, eps, ops._p(acc), ops._p(out), ops._p(coefs), ops._stream(), kernels=2,
                 nbytes=float(B * H * W) * (K * logits.element_size() + 8))
        ctx.save_for_backward(logits, target, coefs)
        ctx.mark_non_differentiable(out)
        return out[0].clone().reshape(()), out

    @staticmethod
    def backward(ctx, g, _gparts):
        logits, target, coefs = ctx.saved_tensors
        B, K, H, W = logits.shape
        gs = g.detach().float().reshape(1).contiguous()
        gl = torch.empty((B, H, W, K), dtype=logits.dtype, device=logits.device)
        ops._run("ce_dice_bwd", ops.lib().unetb200_ce_dice_bwd, ops._p(logits), ops.dt(logits), ops._p(target),
                 B * H * W, K, ops._p(coefs), ops._p(gs), ops._p(gl), ops._stream(),
                 nbytes=float(B * H * W) * (2 * K * logits.element_size() + 8))
        return gl.permute(0, 3, 1, 2), None, None


def ce_dice_loss(logits, target, epsilon=1e-6, return_parts=False):
    """CrossEntropyLoss(logits, target) + dice_loss(softmax(logits).float(), one_hot(target), multiclass=True)
    in one pass over the logits (train.py:137-142).  logits: [B,C,H,W] fp32/bf16, target: int64 [B,H,W]."""
    ops.require_cuda(logits, "ce_dice_loss")
    if logits.dtype not in (torch.float32, torch.bfloat16):
        logits = logits.float()
    K = logits.shape[1]
    lg = logits
    if ops.nhwc_ld(lg) != K:
        lg = logits.contiguous(memory_format=torch.channels_last)
        if ops.nhwc_ld(lg) != K:                  # degenerate sizes: force a packed NHWC copy
            lg = logits.permute(0, 2, 3, 1).contiguous().permute(0, 3, 1, 2)
    tgt = target
    if tgt.dtype != torch.int64 or not tgt.is_contiguous():
        tgt = tgt.long().contiguous()
    total, parts = CeDiceFn.apply(lg, tgt, float(epsilon))
    return (total, parts) if return_parts else total


# ------------------------------------------------------------------------------------------------
# fused BCE + sigmoid dice criterion (the binary branch)
# ------------------------------------------------------------------------------------------------
_TGT_DT = {torch.float32: F32, torch.int64: I64, torch.uint8: U8}


class BceDiceFn(torch.autograd.Function):
    """logits and target in the same (pixel) element order; see :func:`bce_dice_loss`."""

    @staticmethod
    def forward(ctx, logits, target, eps):
        dev = logits.device
        npix = logits.numel()
        L = ops.lib()
        work = torch.empty(L.unetb200_bce_dice_work_bytes(npix), dtype=torch.uint8, device=dev)
        out = torch.empty(4, dtype=torch.float32, device=dev)
        coefs = torch.empty(4, dtype=torch.float32, device=dev)
        ops._run("bce_dice_fwd", L.unetb200_bce_dice_fwd, ops._p(logits), ops.dt(logits), ops._p(target),
                 _TGT_DT[target.dtype], npix, eps, ops._p(work), ops._p(out), ops._p(coefs), ops._stream(), kernels=2,
                 nbytes=float(npix) * (logits.element_size() + target.element_size()))
        ctx.save_for_backward(logits, target, coefs)
        ctx.mark_non_differentiable(out)
        return out[0].clone().reshape(()), out

    @staticmethod
    def backward(ctx, g, _gparts):
        logits, target, coefs = ctx.saved_tensors
        npix = logits.numel()
        gs = g.detach().float().reshape(1).contiguous()
        gl = torch.empty_like(logits)              # a dense layout keeps its strides (same element order)
        ops._run("bce_dice_bwd", ops.lib().unetb200_bce_dice_bwd, ops._p(logits), ops.dt(logits), ops._p(target),
                 _TGT_DT[target.dtype], npix, ops._p(coefs), ops._p(gs), ops._p(gl), ops._stream(),
                 nbytes=float(npix) * (2 * logits.element_size() + target.element_size()))
        return gl, None, None


def bce_dice_loss(logits, target, epsilon=1e-6, return_parts=False):
    """BCEWithLogitsLoss(logits, target) + dice_loss(sigmoid(logits), target) in one pass over the logits: the
    binary branch of train.py:118-134 without its boundary term.  logits: [B,1,H,W] or [B,H,W], fp32 / bf16 (the
    dice term uses the sigmoid rounded to that type, as under autocast); target: [B,H,W] fp32 / int64 / uint8,
    used by value (soft targets allowed).  return_parts: also a device float[4] {total, bce, dice_loss, dice}."""
    ops.require_cuda(logits, "bce_dice_loss")
    if logits.dim() == 4 and logits.size(1) == 1:
        B, _, H, W = logits.shape
    elif logits.dim() == 3:
        B, H, W = logits.shape
    else:
        raise ValueError(f"bce_dice_loss: logits must be [B,1,H,W] or [B,H,W], got {tuple(logits.shape)}")
    if tuple(target.shape) != (B, H, W):
        raise ValueError(f"bce_dice_loss: target {tuple(target.shape)} does not match logits {(B, H, W)}")
    if logits.numel() == 0:
        raise ValueError("bce_dice_loss: empty input")
    lg = logits
    if lg.dtype not in (torch.float32, torch.bfloat16):
        lg = lg.float()
    # one channel: NCHW and channels_last hold the pixels in the same order; anything else is made contiguous
    if not (lg.squeeze(1) if lg.dim() == 4 else lg).is_contiguous():
        lg = lg.contiguous()
    tgt = target
    if tgt.dtype not in _TGT_DT:
        tgt = tgt.float()
    if not tgt.is_contiguous():
        tgt = tgt.contiguous()
    total, parts = BceDiceFn.apply(lg, tgt, float(epsilon))
    return (total, parts) if return_parts else total


# boundary-term constants of the two branches of train.py: (coefficient, edge_width, edge_weight)
_BOUNDARY_BINARY = (0.25, 51, 15)          # train.py:118-134
_BOUNDARY_MULTICLASS = (0.2, 51, 7)        # train.py:143-147 (boundary_weight * norm_factor = 0.2)


def training_criterion(logits, masks, boundary_coeff=None, edge_width=None, edge_weight=None):
    """The loss train.py optimises, branch chosen by the channel count of ``logits``:

    * one channel (n_classes == 1, train.py:118-134): BCEWithLogits + dice(sigmoid) (:func:`bce_dice_loss`)
      + 0.25 * boundary_loss(edge_width=51, edge_weight=15);
    * more (train.py:137-147): CE + multiclass dice (:func:`ce_dice_loss`) + 0.2 * boundary_loss(51, 7).

    ``None`` means that branch's train.py constant; explicit values win and ``boundary_coeff=0`` drops the term.
    Binary masks are used by value: train.py's ``true_masks //= 2`` remap is the caller's."""
    binary = logits.dim() == 4 and logits.size(1) == 1
    d_coeff, d_width, d_weight = _BOUNDARY_BINARY if binary else _BOUNDARY_MULTICLASS
    boundary_coeff = d_coeff if boundary_coeff is None else boundary_coeff
    edge_width = d_width if edge_width is None else edge_width
    edge_weight = d_weight if edge_weight is None else edge_weight
    loss = bce_dice_loss(logits, masks) if binary else ce_dice_loss(logits, masks)
    if boundary_coeff:
        # train.py passes true_masks.float(); the int64 class indices compare identically to 255
        loss = loss + boundary_coeff * boundary_loss(logits, masks, edge_width=edge_width, edge_weight=edge_weight)
    return loss
