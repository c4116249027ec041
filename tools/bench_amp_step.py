"""GradScaler + scheduled tensor LR with FusedRMSprop (train.py:80-85,154-159) on one B200.

    python tools/bench_amp_step.py > profiles/r3_bench_amp_step.json

Prints one JSON line with the GPU name and power limit read in the same run, and:

* the optimizer side of an eager step over the 31 036 546 parameters of UNet(1, 2) (64 fp32 tensors, 124 MB each of
  weights, gradients, square_avg and momentum_buffer: every pass reads HBM), from scaled gradients to the updated
  weights, for
  - ``torch_foreach``: torch.optim.RMSprop(foreach=True) in train.py's order: ``unscale_``, ``clip_grad_norm_``,
    ``scaler.step`` (GradScaler decides on the host: one sync per step), ``scaler.update``;
  - ``fused_train_py_order``: the same calls on FusedRMSprop with a tensor lr (no sync);
  - ``fused_folded``: ``scaler.step(opt, clip_max_norm=1.0)`` + ``update`` on FusedRMSprop with a tensor lr;
  - ``fused_no_scaler``: ``opt.step(clip_max_norm=1.0)`` with a float lr, the step without GradScaler.
  Host wall time per call ending in a device synchronise (what an eager loop pays), and device time between CUDA
  events around the same calls, median of rounds that alternate the arms.  Gradients are refreshed, untimed, before
  each call.
* graphed UNet(1, 2) training img/s at B = 16, 512x512, bf16 autocast: today's captured step (FusedRMSprop with a
  float lr, ``opt.step(clip_max_norm=1.0)``) against the captured step with GradScaler and a tensor lr
  (``scaler.scale(loss).backward()``, ``scaler.step(opt, clip_max_norm=1.0)``, ``scaler.update()``), replayed
  back to back and with ``CosineAnnealingWarmRestarts.step()`` between replays; interleaved rounds.
"""
import json
import os
import statistics
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "unet-medical-image-contour-segmentation_b200"))
import unet  # noqa: E402
from unetb200 import losses as UL  # noqa: E402
from unetb200.graph import GraphedStep  # noqa: E402
from unetb200.optim import FusedRMSprop  # noqa: E402

B, S = 16, 512
dev = torch.device("cuda:0")
HYPER = dict(alpha=0.99, eps=1e-8, weight_decay=1e-8, momentum=0.999)      # train.py:80-84


def gpu_info():
    info = {"gpu": torch.cuda.get_device_name(dev)}
    try:
        info["power_limit_and_max_sm_clock"] = subprocess.check_output(
            ["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
            text=True).strip()
    except (OSError, subprocess.CalledProcessError) as exc:
        info["power_limit_and_max_sm_clock"] = f"unavailable: {exc}"
    return info


def optimizer_side(iters=40, rounds=3):
    torch.manual_seed(0)
    weights = [p.detach().to(dev) for p in unet.UNet(1, 2).parameters()]
    gen = torch.Generator(device=dev).manual_seed(1)
    grads = [torch.randn(w.shape, device=dev, generator=gen) * 1e-2 for w in weights]

    def arm(kind):
        ps = [torch.nn.Parameter(w.clone()) for w in weights]
        if kind == "torch_foreach":
            opt = torch.optim.RMSprop(ps, lr=1e-5, foreach=True, **HYPER)
        elif kind == "fused_no_scaler":
            opt = FusedRMSprop(ps, lr=1e-5, **HYPER)
        else:
            opt = FusedRMSprop(ps, lr=torch.tensor(1e-5, device=dev), **HYPER)
        scaler = torch.amp.GradScaler("cuda")
        scaler.scale(torch.ones((), device=dev))       # creates the scale tensor (65536), as the loss's scale() does
        for p in ps:
            p.grad = torch.empty_like(p)
        src = [g * 65536.0 for g in grads] if kind != "fused_no_scaler" else grads

        def call():
            if kind == "fused_no_scaler":
                opt.step(clip_max_norm=1.0)
                return
            if kind == "fused_folded":
                scaler.step(opt, clip_max_norm=1.0)
            else:
                scaler.unscale_(opt)
                torch.nn.utils.clip_grad_norm_(ps, 1.0)
                scaler.step(opt)
            scaler.update()
        return ps, src, call

    kinds = ("torch_foreach", "fused_train_py_order", "fused_folded", "fused_no_scaler")
    arms = {k: arm(k) for k in kinds}
    res = {k: {"host_ms": [], "device_ms": []} for k in kinds}
    for r in range(rounds + 1):                    # round 0 warms every arm up and is dropped
        for k in kinds:
            ps, src, call = arms[k]
            host, device = [], []
            for _ in range(iters):
                torch._foreach_copy_([p.grad for p in ps], src)
                torch.cuda.synchronize()
                s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                t0 = time.perf_counter()
                s.record()
                call()
                e.record()
                torch.cuda.synchronize()
                host.append((time.perf_counter() - t0) * 1e3)
                device.append(s.elapsed_time(e))
            if r:
                res[k]["host_ms"].append(statistics.median(host))
                res[k]["device_ms"].append(statistics.median(device))
    out = {"workload": f"{sum(w.numel() for w in weights)} fp32 parameters in {len(weights)} tensors (UNet(1,2)), "
                       f"clip 1.0, eager; median of {iters} calls per round, {rounds} alternating rounds"}
    for k in kinds:
        out[k] = {"host_ms_rounds": res[k]["host_ms"], "device_ms_rounds": res[k]["device_ms"],
                  "host_ms": statistics.median(res[k]["host_ms"]),
                  "device_ms": statistics.median(res[k]["device_ms"])}
    return out


def train_steps(reps=30, rounds=3):
    torch.manual_seed(0)
    img = torch.rand(B, 1, S, S, device=dev).contiguous(memory_format=torch.channels_last)
    msk = torch.randint(0, 2, (B, S, S), device=dev)
    state = {k: v.clone() for k, v in unet.UNet(1, 2).state_dict().items()}
    steps, scheds = {}, {}
    for kind in ("float_lr_no_scaler", "grad_scaler_tensor_lr"):
        model = unet.UNet(1, 2)
        model.load_state_dict(state)
        model = model.to(dev).to(memory_format=torch.channels_last).train()
        if kind == "float_lr_no_scaler":
            opt = FusedRMSprop(model.parameters(), lr=1e-5, **HYPER)
            scaler = None
        else:
            opt = FusedRMSprop(model.parameters(), lr=torch.tensor(1e-5, device=dev), **HYPER)
            scaler = torch.amp.GradScaler("cuda")
            scheds[kind] = torch.optim.lr_scheduler.CosineAnnealingWarmRestarts(opt, T_0=5)

        def step(x, t, model=model, opt=opt, scaler=scaler):
            opt.zero_grad(set_to_none=True)
            with torch.autocast("cuda", enabled=True):
                loss = UL.training_criterion(model(x), t, boundary_coeff=0.2, edge_width=51, edge_weight=7)
            if scaler is None:
                loss.backward()
                opt.step(clip_max_norm=1.0)
            else:
                scaler.scale(loss).backward()
                scaler.step(opt, clip_max_norm=1.0)
                scaler.update()
            return loss
        steps[kind] = GraphedStep(step, (img, msk), warmup=2)

    def timed(g, sched):
        for _ in range(3):
            g.replay()
        torch.cuda.synchronize()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(reps):
            g.replay()
            if sched is not None:
                sched.step()
        e.record()
        torch.cuda.synchronize()
        ms = s.elapsed_time(e) / reps
        return {"ms_per_step": ms, "img_per_s": B * 1e3 / ms}

    arms = {"float_lr_no_scaler": (steps["float_lr_no_scaler"], None),
            "grad_scaler_tensor_lr": (steps["grad_scaler_tensor_lr"], None),
            "grad_scaler_tensor_lr_with_scheduler_step": (steps["grad_scaler_tensor_lr"],
                                                          scheds["grad_scaler_tensor_lr"])}
    res = {k: [] for k in arms}
    for _ in range(rounds):
        for k, (g, sched) in arms.items():
            res[k].append(timed(g, sched))
    finite = {k: bool(torch.isfinite(g.static_loss).item()) for k, g in steps.items()}
    out = {"workload": f"UNet(1,2) B={B} {S}x{S}, bf16 autocast, whole-step CUDA graph, clip 1.0, {reps} replays per "
                       f"round, {rounds} interleaved rounds",
           "steps": res, "loss_finite": finite}
    best = {k: max(r["img_per_s"] for r in v) for k, v in res.items()}
    out["best_img_per_s"] = best
    out["scaler_over_no_scaler"] = best["grad_scaler_tensor_lr"] / best["float_lr_no_scaler"]
    out["scaler_with_scheduler_over_no_scaler"] = (best["grad_scaler_tensor_lr_with_scheduler_step"]
                                                   / best["float_lr_no_scaler"])
    return out


def main():
    assert torch.cuda.is_available(), "tools/bench_amp_step.py measures on a CUDA device"
    torch.cuda.set_device(dev)
    line = gpu_info()
    line["optimizer_side"] = optimizer_side()
    line["train_step"] = train_steps()
    print(json.dumps(line))


if __name__ == "__main__":
    main()
