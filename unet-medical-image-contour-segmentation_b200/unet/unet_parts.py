"""B200-native drop-ins for the reference's ``unet/unet_parts.py`` (same class names, constructor
signatures, sub-module names and therefore the same ``state_dict`` keys).

The ``nn.Conv2d`` / ``nn.BatchNorm2d`` / ``nn.ConvTranspose2d`` children are *parameter holders only*:
they give the reference's key names (``double_conv.0.weight`` ...), shapes and default initialisation
(so ``torch.manual_seed(s); UNet(...)`` draws the reference's weights), but their ``forward`` is never
called.  ``forward`` here dispatches to the autograd Functions of ``unetb200.functional`` which run
hand-written sm_100a kernels through the C ABI; there is no cuDNN/ATen and no CPU fallback.
"""
import torch
import torch.nn as nn

from unetb200 import backward_pass, ops
from unetb200 import functional as UF
from unetb200.functional import _Cfg


def _to_internal(x, dtype):
    """NHWC of `dtype`, keeping the autograd graph when the caller's tensor needs a gradient."""
    if x.dtype == dtype and ops.nhwc_ld(x) is not None:
        return x
    if x.requires_grad and torch.is_grad_enabled():
        return UF.ToNHWCFn.apply(x, dtype)
    return ops.to_nhwc(x, dtype)


def _prep(x, what):
    """Caller tensor (fp32 NCHW-logical, usually channels_last) -> NHWC of the compute dtype."""
    ops.require_cuda(x, what)
    backward_pass.begin_forward()
    if x.dim() != 4:
        raise ValueError(f"{what}: expected a [B, C, H, W] tensor, got {tuple(x.shape)}")
    return _to_internal(x, UF.compute_dtype(x))


def _needs_graph(module, *tensors):
    return torch.is_grad_enabled() and (any(t.requires_grad for t in tensors) or
                                        any(p.requires_grad for p in module.parameters()))


class DoubleConv(nn.Module):
    """(conv3x3 pad 1, no bias -> BatchNorm2d -> ReLU) twice  [reference unet_parts.py:7-24]."""

    def __init__(self, in_channels, out_channels, mid_channels=None):
        super().__init__()
        mid = mid_channels if mid_channels else out_channels
        holders = [nn.Conv2d(in_channels, mid, kernel_size=3, padding=1, bias=False), nn.BatchNorm2d(mid),
                   nn.ReLU(inplace=True),
                   nn.Conv2d(mid, out_channels, kernel_size=3, padding=1, bias=False), nn.BatchNorm2d(out_channels),
                   nn.ReLU(inplace=True)]
        self.double_conv = nn.Sequential(*holders)

    def run(self, x, out=None, want_pool=False, outconv=None):
        """x: NHWC compute-dtype tensor.  Returns z or (z, maxpool2(z)); ``out`` = optional
        caller-owned destination (a channel slice of a concat buffer).  ``outconv`` = the OutConv module that follows
        directly (inference only): when the fused kernel covers the shape the return value is ``(logits, True)``,
        else ``(z, False)``."""
        c1, bn1, _, c2, bn2, _ = self.double_conv
        if x.shape[1] != c1.in_channels:
            raise ValueError(f"DoubleConv expects {c1.in_channels} input channels, got {x.shape[1]}")
        cfg = _Cfg(bn1=bn1, bn2=bn2, training=self.training, out=out, want_pool=want_pool,
                   save=_needs_graph(self, x))
        if outconv is not None:
            if not cfg.save and not _needs_graph(outconv, x):
                cfg.outconv = (outconv.conv.weight.detach(), outconv.conv.bias.detach() if outconv.conv.bias is not None else None)
            res = UF.DoubleConvFn.apply(x, c1.weight, bn1.weight, bn1.bias, c2.weight, bn2.weight, bn2.bias, cfg)
            return res, bool(getattr(cfg, "fused_outconv", False))
        return UF.DoubleConvFn.apply(x, c1.weight, bn1.weight, bn1.bias, c2.weight, bn2.weight, bn2.bias, cfg)

    def forward(self, x):
        return self.run(_prep(x, "DoubleConv"))


class Down(nn.Module):
    """MaxPool2d(2) then DoubleConv  [reference unet_parts.py:26-37]."""

    def __init__(self, in_channels, out_channels):
        super().__init__()
        self.maxpool_conv = nn.Sequential(nn.MaxPool2d(2), DoubleConv(in_channels, out_channels))

    def run(self, pooled, out=None, want_pool=False):
        """``pooled`` is the already max-pooled input (fused into the producer's BN-apply kernel)."""
        return self.maxpool_conv[1].run(pooled, out=out, want_pool=want_pool)

    def forward(self, x):
        x = _prep(x, "Down")
        if x.shape[2] < 2 or x.shape[3] < 2:
            raise ValueError(f"Down: input {tuple(x.shape)} is too small for MaxPool2d(2)")
        return self.maxpool_conv[1].run(UF.MaxPoolFn.apply(x))


class SpatialAttention(nn.Module):
    """sigmoid(conv7x7([mean_c x, max_c x]))  [reference unet_parts.py:39-60].  ``forward`` returns the attention map
    like the reference; ``gate`` applies it (x * map, unet_parts.py:91-92) in the same kernels."""

    def __init__(self, kernel_size=7):
        super().__init__()
        assert kernel_size in (3, 7), "kernel size must be 3 or 7"
        if kernel_size != 7:
            raise NotImplementedError("unetb200: SpatialAttention(kernel_size=3) is never built by the reference models "
                                      "(unet_parts.py:77 uses the default 7) and has no kernel here")
        self.conv1 = nn.Conv2d(2, 1, kernel_size, padding=3, bias=False)
        self.sigmoid = nn.Sigmoid()

    def gate(self, x, out=None):
        """x: NHWC compute-dtype tensor -> x * attention(x), optionally written into ``out``."""
        cfg = _Cfg(out=out, save=_needs_graph(self, x))
        return UF.SpatialGateFn.apply(x, self.conv1.weight, cfg)

    def forward(self, x):
        raise NotImplementedError("unetb200: the bare attention map is not exposed -- the reference only ever uses it as "
                                  "x2 * attention(x2) (Up.forward, unet_parts.py:91-92), which is SpatialAttention.gate(x)")


class Up(nn.Module):
    """Upsample x1 (ConvTranspose2d k2 s2, or bilinear x2 align_corners=True), pad to x2, cat([x2, x1]),
    DoubleConv  [reference unet_parts.py:62-98]."""

    def __init__(self, in_channels, out_channels, bilinear=True, use_attention=False):
        super().__init__()
        if bilinear:
            self.up = nn.Upsample(scale_factor=2, mode="bilinear", align_corners=True)
            self.conv = DoubleConv(in_channels, out_channels, in_channels // 2)
        else:
            self.up = nn.ConvTranspose2d(in_channels, in_channels // 2, kernel_size=2, stride=2)
            self.conv = DoubleConv(in_channels, out_channels)
        self.bilinear = bilinear
        self.use_attention = use_attention
        self.attention = SpatialAttention() if use_attention else nn.Identity()      # unet_parts.py:76-77

    def run(self, x1, x2, cat=None, out=None, want_pool=False, outconv=None):
        """x2: the skip tensor.  With attention it is the UN-gated encoder output (kept for the gate's backward); the
        gated copy is written into the skip half of ``cat`` when the caller pre-allocated the concat buffer."""
        if self.use_attention:                         # unet_parts.py:91-92
            dst = ops.channel_slice(cat, 0, x2.shape[1]) if cat is not None else None
            x2 = self.attention.gate(x2, out=dst)
        cfg = _Cfg(cat=cat, save=_needs_graph(self, x1, x2))
        if self.bilinear:
            merged = UF.UpCatBilinearFn.apply(x1, x2, cfg)
        else:
            merged = UF.UpCatConvTFn.apply(x1, x2, self.up.weight, self.up.bias, cfg)
        if outconv is not None:
            return self.conv.run(merged, out=out, want_pool=want_pool, outconv=outconv)
        return self.conv.run(merged, out=out, want_pool=want_pool)

    def forward(self, x1, x2):
        x1 = _prep(x1, "Up")
        ops.require_cuda(x2, "Up")
        return self.run(x1, _to_internal(x2, x1.dtype))


class OutConv(nn.Module):
    """1x1 conv with bias  [reference unet_parts.py:100-106]."""

    def __init__(self, in_channels, out_channels):
        super().__init__()
        self.conv = nn.Conv2d(in_channels, out_channels, kernel_size=1)

    def run(self, x):
        cfg = _Cfg(save=_needs_graph(self, x))
        return UF.OutConvFn.apply(x, self.conv.weight, self.conv.bias, cfg)

    def forward(self, x):
        return self.run(_prep(x, "OutConv"))
