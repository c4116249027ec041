"""B200-native drop-in for the reference's ``unet/unet_model.py``: ``UNet(n_channels, n_classes,
bilinear=False)`` with the reference's attributes, sub-module names and ``state_dict`` layout
(reference unet_model.py:8-50), plus the width variants ``UNet_S`` / ``UNet_T`` that train.py imports.

``forward`` runs the whole network on hand-written sm_100a kernels (see ``unetb200``): activations are
NHWC in the compute dtype (bf16 under autocast, else fp32), every encoder stage writes its skip
tensor straight into the first half of the decoder's concat buffer and emits its 2x2 max-pool from
the same kernel, and the upsampling kernels write the second half -- ``torch.cat`` and
``nn.MaxPool2d`` never run as separate passes.
"""
import logging

import torch
import torch.nn as nn

from unetb200 import ops

from .unet_parts import DoubleConv, Down, OutConv, Up, _prep


class _UNetBase(nn.Module):
    _BASE = 64
    _ATTENTION = False    # UNet_SA: SpatialAttention gate on every skip tensor (unet_model.py:156-160)
    _taps = None          # dict to fill with the named intermediate tensors of the next forward, or None

    def __init__(self, n_channels, n_classes, bilinear=False):
        super().__init__()
        self.n_channels = n_channels
        self.n_classes = n_classes
        self.bilinear = bilinear
        b = self._BASE
        factor = 2 if bilinear else 1
        self.inc = DoubleConv(n_channels, b)
        self.down1 = Down(b, 2 * b)
        self.down2 = Down(2 * b, 4 * b)
        self.down3 = Down(4 * b, 8 * b)
        self.down4 = Down(8 * b, 16 * b // factor)
        att = self._ATTENTION
        self.up1 = Up(16 * b, 8 * b // factor, bilinear, use_attention=att)
        self.up2 = Up(8 * b, 4 * b // factor, bilinear, use_attention=att)
        self.up3 = Up(4 * b, 2 * b // factor, bilinear, use_attention=att)
        self.up4 = Up(2 * b, b, bilinear, use_attention=att)
        self.outc = OutConv(b, n_classes)

    def forward(self, x):
        from unetb200 import functional as UF
        if self._bn_doubles is None:
            from unetb200 import ddp
            ddp.sync_bn_process_group(self, self.training)      # raises for mixed process groups
            self._bn_doubles = self.bn_arena_doubles()
        with UF.zero_arena(self._bn_doubles if self.training else 0, x.device):
            return self._forward(x)

    _bn_doubles = None

    def bn_arena_doubles(self):
        """Size of the fp64 statistics arena of a training forward: 2 C accumulators (sum, sum of squares) per
        BatchNorm holder -- BatchNorm2d, or the nn.SyncBatchNorm that convert_sync_batchnorm puts in its place."""
        return sum(2 * ((m.num_features + 1) // 2 * 2) for m in self.modules()
                   if isinstance(m, nn.modules.batchnorm._BatchNorm))

    def _forward(self, x):
        x = _prep(x, type(self).__name__)
        B, C, H, W = x.shape
        if C != self.n_channels:
            raise ValueError(f"{type(self).__name__} was built for {self.n_channels} input channels, got {C}")
        if H < 16 or W < 16:
            raise ValueError(f"{type(self).__name__}: input {H}x{W} is too small for four 2x2 max-pools")
        b = self._BASE
        dev, cd = x.device, x.dtype
        from unetb200 import functional as UF
        UF.prepack(self, cd, need_dgrad=torch.is_grad_enabled())
        # concat buffers of the four Up stages: [skip | upsampled], at the skip's resolution
        cats = [ops.empty_nhwc(B, 2 * b * (1 << k), H >> k, W >> k, cd, dev) for k in range(4)]
        # (with attention the encoder keeps its own un-gated output -- the gate's backward needs it -- and the gate
        # writes x * attention(x) into the skip half of the concat buffer)
        skips = [None if self._ATTENTION else ops.channel_slice(cats[k], 0, b * (1 << k)) for k in range(4)]
        taps = self._taps
        cut = UF.CutFn.apply if taps is not None else (lambda t: t)
        ck = self._stage if (self._checkpointing and taps is None and torch.is_grad_enabled()) else (lambda fn, *t: fn(*t))
        x1, p = ck(lambda t: self.inc.run(t, out=skips[0], want_pool=True), x)
        x2, p = ck(lambda t: self.down1.run(t, out=skips[1], want_pool=True), p)
        x3, p3 = ck(lambda t: self.down2.run(t, out=skips[2], want_pool=True), p)
        p3c = cut(p3)
        x4, p = ck(lambda t: self.down3.run(t, out=skips[3], want_pool=True), p3c)
        x5 = ck(lambda t: self.down4.run(t), p)
        x5c, x4c, x3c = cut(x5), cut(x4), cut(x3)
        y = ck(lambda a, b_: self.up1.run(a, b_, cat=cats[3]), x5c, x4c)
        u2 = ck(lambda a, b_: self.up2.run(a, b_, cat=cats[2]), y, x3c)
        u2c, x2c, x1c = cut(u2), cut(x2), cut(x1)
        y = ck(lambda a, b_: self.up3.run(a, b_, cat=cats[1]), u2c, x2c)
        if not torch.is_grad_enabled() and not self.training:
            # inference: OutConv rides in the epilogue of the last conv when the fused kernel covers the shape
            y, fused = self.up4.run(y, x1c, cat=cats[0], outconv=self.outc)
            out = y if fused else self.outc.run(y)
        else:
            y = ck(lambda a, b_: self.up4.run(a, b_, cat=cats[0]), y, x1c)
            out = self.outc.run(y)
        if taps is not None:
            # cut points of a segmented backward pass (unetb200.ddp.SegmentedStep): name -> (tensor, its cut alias)
            taps.update(x1=(x1, x1c), x2=(x2, x2c), x3=(x3, x3c), x4=(x4, x4c), x5=(x5, x5c), p3=(p3, p3c),
                        u2=(u2, u2c))
        return out

    _checkpointing = False

    @staticmethod
    def _stage(fn, *tensors):
        """One encoder / decoder stage under activation re-computation: only the stage's inputs stay resident, its raw
        conv outputs and inner activations are re-computed (by the same deterministic kernels: bit-identical) when the
        backward pass reaches it.  BatchNorm running statistics move once (functional.recompute_mode)."""
        from contextlib import nullcontext

        from torch.utils.checkpoint import checkpoint
        from unetb200 import functional as UF
        return checkpoint(fn, *tensors, use_reentrant=False, preserve_rng_state=False,
                          context_fn=lambda: (nullcontext(), UF.recompute_mode()))

    def use_checkpointing(self):
        """Called by train.py:299 after a CUDA OOM: from the next forward on every DoubleConv / Down / Up stage is run
        under activation re-computation (what the reference's unet_model.py:40-50 intends; its own implementation
        raises TypeError because it calls checkpoint() without inputs).  Trades one extra forward pass of the stage
        inside backward for ~2/3 of the saved activations; results are unchanged."""
        logging.info("unetb200: activation re-computation enabled for the encoder / decoder stages")
        self._checkpointing = True


class UNet(_UNetBase):
    """Standard UNet, widths 64-128-256-512-1024 (reference unet_model.py:8-38)."""
    _BASE = 64


class UNet_S(_UNetBase):
    """Light variant, base width 16 (reference unet_model.py:96-138)."""
    _BASE = 16


class UNet_T(_UNetBase):
    """Tiny variant, base width 8 (reference unet_model.py:52-94)."""
    _BASE = 8


class UNet_SA(_UNetBase):
    """UNet with a SpatialAttention gate on every skip connection, base width 16 (reference unet_model.py:140-189)."""
    _BASE = 16
    _ATTENTION = True
