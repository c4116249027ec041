"""Fused optimizer step for the UNet training loop: clip_grad_norm_ + RMSprop in two multi-tensor kernels.

``FusedRMSprop`` has torch.optim.RMSprop's constructor, ``state_dict`` layout (``step``, ``square_avg``,
``momentum_buffer``) and arithmetic (reference train.py:80-84); ``step(clip_max_norm=...)`` additionally folds
``torch.nn.utils.clip_grad_norm_(params, max_norm)`` (train.py:157) into the same pass.  All 64 parameter
tensors are updated by one launch each of ``unetb200_grad_sqnorm`` and ``unetb200_rmsprop_step`` instead of
~25 foreach launches; capture-safe (no host sync).

Captured steps with torch.amp.GradScaler and LR schedulers (train.py:80-85,154-159): ``lr`` may be a 0-dim fp32
CUDA tensor, which the kernel reads on the device, so a graph replay uses whatever a scheduler wrote into it
between replays (a float ``lr`` is a kernel argument, fixed when the step is captured).  The optimizer sets
``_step_supports_amp_scaling``: ``GradScaler.step`` hands it ``grad_scale`` / ``found_inf`` tensors instead of
deciding on the host, and the step unscales, checks, clips and updates on the device (``unetb200_grad_sqnorm_amp``
+ ``unetb200_rmsprop_step_amp``), storing nothing when an inf / NaN was found.
"""
from __future__ import annotations

import ctypes as C

import torch

from . import backward_pass, ops


def _dense(t):
    """Non-overlapping and dense: the strides are a permutation of a contiguous layout."""
    expect = 1
    for st, sz in sorted((st, sz) for sz, st in zip(t.shape, t.stride()) if sz > 1):
        if st != expect:
            return False
        expect *= sz
    return True


def _check_hyper(group):
    """lr: a float or a 0-dim fp32 CUDA tensor; every other hyper-parameter a number (the kernels take them as
    launch arguments)."""
    for k in ("alpha", "eps", "weight_decay", "momentum"):
        if isinstance(group[k], torch.Tensor):
            raise ValueError(f"FusedRMSprop: {k} must be a number, not a tensor (only lr may be a tensor)")
    lr = group["lr"]
    if not isinstance(lr, torch.Tensor):
        return
    if lr.dim() != 0:
        raise ValueError(f"FusedRMSprop: a tensor lr must be 0-dim (got shape {tuple(lr.shape)})")
    if lr.dtype != torch.float32:
        raise ValueError(f"FusedRMSprop: a tensor lr must be float32 (got {lr.dtype})")
    if not lr.is_cuda:
        raise ValueError(f"FusedRMSprop: a tensor lr must be a CUDA tensor (got one on {lr.device})")


class FusedRMSprop(torch.optim.Optimizer):
    # GradScaler.step passes grad_scale / found_inf as attributes instead of syncing to decide on the host
    _step_supports_amp_scaling = True

    def __init__(self, params, lr=1e-2, alpha=0.99, eps=1e-8, weight_decay=0, momentum=0, centered=False,
                 capturable=True, foreach=None, maximize=False, differentiable=False):
        if centered or maximize or differentiable:
            raise NotImplementedError("FusedRMSprop: centered / maximize / differentiable are not implemented")
        hyper = dict(lr=lr, alpha=alpha, eps=eps, weight_decay=weight_decay, momentum=momentum)
        _check_hyper(hyper)
        if lr < 0 or eps < 0 or momentum < 0 or weight_decay < 0 or alpha < 0:
            raise ValueError("FusedRMSprop: negative hyper-parameter")
        super().__init__(params, dict(hyper, centered=False, capturable=capturable, foreach=foreach, maximize=False,
                                      differentiable=False))
        self._norm = None

    def _tables(self, tensors_lists):
        n = len(tensors_lists[0])
        arrs = []
        for lst in tensors_lists:
            if lst is None:
                arrs.append(None)
                continue
            a = (C.c_void_p * n)(*[t.data_ptr() for t in lst])
            arrs.append(a)
        numel = (C.c_int64 * n)(*[t.numel() for t in tensors_lists[0]])
        return arrs, numel, n

    @torch.no_grad()
    def step(self, closure=None, clip_max_norm=None, write_clipped_grad=True):
        """One update.  clip_max_norm: fold clip_grad_norm_(all params of this optimizer, clip_max_norm) in;
        returns the total gradient norm (a 0-dim device tensor) in that case, else the closure's loss.  Like
        clip_grad_norm_ (train.py:157) the clipped gradients are written back to ``p.grad`` (same pass, one more
        store per element); ``write_clipped_grad=False`` leaves ``p.grad`` unclipped.

        Under ``GradScaler.step(opt, ...)`` the attributes ``grad_scale`` (the scale, or None after ``unscale_``)
        and ``found_inf`` are set: gradients are unscaled in the kernels, the norm is that of the unscaled
        gradients, and a non-zero found_inf leaves parameters, state and gradients untouched.  With ``grad_scale``
        and no ``found_inf`` (a direct call) the norm pass also computes the flag.  No host synchronisation."""
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        grad_scale = getattr(self, "grad_scale", None)
        found_inf = getattr(self, "found_inf", None)
        amp = grad_scale is not None or found_inf is not None
        groups = []
        all_grads = []
        steps = []
        for group in self.param_groups:
            _check_hyper(group)
            amp = amp or isinstance(group["lr"], torch.Tensor)
            ps, gs, sqs, moms, group_steps = [], [], [], [], []
            for p in group["params"]:
                if p.grad is None:
                    continue
                ops.require_cuda(p, "FusedRMSprop")
                if p.dtype != torch.float32 or p.grad.dtype != torch.float32:
                    raise ValueError("FusedRMSprop: fp32 parameters and gradients only")
                st = self.state[p]
                if len(st) == 0:
                    st["step"] = torch.zeros((), dtype=torch.float32, device=p.device)
                    st["square_avg"] = torch.zeros_like(p, memory_format=torch.preserve_format)
                    if group["momentum"] > 0:
                        st["momentum_buffer"] = torch.zeros_like(p, memory_format=torch.preserve_format)
                g = p.grad
                # the kernel walks raw storage: all four tensors must share one dense element order
                if g.stride() != p.stride():          # re-layout into a temporary; p.grad itself is left alone
                    g = torch.empty_like(p, memory_format=torch.preserve_format).copy_(g)
                if st["square_avg"].stride() != p.stride() or not _dense(p):
                    raise ValueError("FusedRMSprop: parameters must be dense and state must share their layout")
                if isinstance(group["lr"], torch.Tensor) and group["lr"].device != p.device:
                    raise ValueError(f"FusedRMSprop: lr is on {group['lr'].device}, a parameter on {p.device}")
                group_steps.append(st["step"])
                ps.append(p)
                gs.append(g)
                sqs.append(st["square_avg"])
                if group["momentum"] > 0:
                    moms.append(st["momentum_buffer"])
            if ps:
                groups.append((group, ps, gs, sqs, moms if group["momentum"] > 0 else None, group_steps))
                all_grads += gs
                steps += group_steps
        if not groups:
            return loss
        if amp:
            norm = self._step_amp(groups, all_grads, clip_max_norm, write_clipped_grad, grad_scale, found_inf)
            return norm if clip_max_norm is not None else loss
        torch._foreach_add_(steps, 1)                  # one launch for all step counters
        backward_pass.side_stream_sync()
        norm = None
        sumsq = None
        if clip_max_norm is not None:
            sumsq = torch.empty(1, dtype=torch.float64, device=all_grads[0].device)
            (ga,), numel, n = self._tables([all_grads])
            ops._run("grad_sqnorm", ops.lib().unetb200_grad_sqnorm, ga, numel, n, ops._p(sumsq), ops._stream(),
                     nbytes=4.0 * sum(g.numel() for g in all_grads))
            norm = sumsq.sqrt().float().reshape(())
        for group, ps, gs, sqs, moms, _ in groups:
            (wa, ga, sa, ma), numel, n = self._tables([ps, gs, sqs, moms])
            ops._run("rmsprop_step", ops.lib().unetb200_rmsprop_step, wa, ga, sa, ma, numel, n,
                     ops._p(sumsq) if sumsq is not None else C.c_void_p(0),
                     float(clip_max_norm) if clip_max_norm is not None else 0.0, float(group["lr"]),
                     float(group["alpha"]), float(group["eps"]), float(group["weight_decay"]), float(group["momentum"]),
                     1 if (clip_max_norm is not None and write_clipped_grad) else 0, ops._stream(),
                     nbytes=4.0 * sum(p.numel() for p in ps) * (7 if moms else 5))
            # the kernel writes through raw pointers: tell autograd (saved-tensor checks) and the packed-operand
            # cache of unetb200.functional that these tensors changed
            torch._C._increment_version(ps)
        return norm if clip_max_norm is not None else loss

    def _step_amp(self, groups, all_grads, clip_max_norm, write_clipped_grad, grad_scale, found_inf):
        """The device-side step: lr, 1/grad_scale and found_inf are read by the kernels, step counters move only
        when the step is taken."""
        backward_pass.side_stream_sync()
        dev = all_grads[0].device
        inv_scale = None
        if grad_scale is not None:
            inv_scale = grad_scale.double().reciprocal().float()       # as GradScaler.unscale_ computes it
        if found_inf is not None and (found_inf.numel() != 1 or found_inf.dtype != torch.float32):
            raise ValueError("FusedRMSprop: found_inf must be a one-element float32 tensor")
        check = grad_scale is not None and found_inf is None          # opt.step() called directly with a scale
        if check:
            found_inf = torch.zeros((), dtype=torch.float32, device=dev)
        norm = None
        sumsq = None
        if clip_max_norm is not None:
            sumsq = torch.empty(1, dtype=torch.float64, device=dev)
        if sumsq is not None or check:
            (ga,), numel, n = self._tables([all_grads])
            ops._run("grad_sqnorm_amp", ops.lib().unetb200_grad_sqnorm_amp, ga, numel, n, ops._p(inv_scale),
                     ops._p(sumsq), ops._p(found_inf) if check else C.c_void_p(0), ops._stream(),
                     nbytes=4.0 * sum(g.numel() for g in all_grads))
        if sumsq is not None:
            norm = sumsq.sqrt().float().reshape(())
        for group, ps, gs, sqs, moms, group_steps in groups:
            lr = group["lr"]
            if not isinstance(lr, torch.Tensor):                     # fixed at capture, like the float path
                lr = torch.full((), float(lr), dtype=torch.float32, device=dev)
            (wa, ga, sa, ma, ta), numel, n = self._tables([ps, gs, sqs, moms, group_steps])
            ops._run("rmsprop_step_amp", ops.lib().unetb200_rmsprop_step_amp, wa, ga, sa, ma, ta, numel, n,
                     ops._p(sumsq), float(clip_max_norm) if clip_max_norm is not None else 0.0, ops._p(lr),
                     ops._p(inv_scale), ops._p(found_inf), float(group["alpha"]), float(group["eps"]),
                     float(group["weight_decay"]), float(group["momentum"]),
                     1 if (clip_max_norm is not None and write_clipped_grad) else 0, ops._stream(),
                     nbytes=4.0 * sum(p.numel() for p in ps) * (7 if moms else 5))
            torch._C._increment_version(ps)
        return norm
