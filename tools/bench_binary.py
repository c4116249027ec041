"""Binary (n_classes = 1, train.py:118-134) criterion and training step on one B200.

    python tools/bench_binary.py > profiles/r3_bench_binary.json

Prints one JSON line with the GPU name and power limit read in the same run, and:

* criterion forward + backward device time at B = 16, 512x512, bf16 logits (the autocast output of OutConv),
  fp32 {0,1} targets, for (a) the fused BCE + dice kernel pair alone, (b) the whole binary criterion
  ``losses.training_criterion`` (fused pair + boundary term) and (c) the chain train.py:118-134 runs on the drop-in
  modules today: ATen BCE-with-logits and sigmoid, ``utils.dice_score.dice_loss``, ``utils.boundary_loss``.  Each
  pass over more than twice the 126 MB L2 of distinct input sets is captured in a CUDA graph and replayed (CUDA
  events), so every launch reads HBM and no Python time hides the kernels.  GB/s are the algorithmic bytes of the
  fused design (2 + 4 B per pixel forward, 2 + 4 + 2 backward, 2 + 4 for the boundary pass) over the time, against
  the measured 6 530 GB/s copy peak.  Launches are counted with torch.profiler on one eager call.
* whole-step CUDA-graph training img/s for UNet(1,1) / UNet_S(1,1) (binary criterion defaults) next to UNet(1,2) /
  UNet_S(1,2) (the 2-class criterion bench.py times), FusedRMSprop + clip as in bench.py, two interleaved rounds.
"""
import json
import os
import subprocess
import sys

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "unet-medical-image-contour-segmentation_b200"))
import unet.unet_model as UM  # noqa: E402
from unetb200 import losses as UL  # noqa: E402
from unetb200 import ops  # noqa: E402
from unetb200.graph import GraphedStep  # noqa: E402
from unetb200.optim import FusedRMSprop  # noqa: E402
from utils.boundary_loss import boundary_loss  # noqa: E402
from utils.dice_score import dice_loss  # noqa: E402

PEAK = 6530.3          # GB/s, measured copy peak (DESIGN.md section 3.2)
L2_BYTES = 126e6
B, S = 16, 512
dev = torch.device("cuda:0")


def gpu_info():
    info = {"gpu": torch.cuda.get_device_name(dev)}
    try:
        info["power_limit_and_max_sm_clock"] = subprocess.check_output(
            ["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
            text=True).strip()
    except (OSError, subprocess.CalledProcessError) as exc:
        info["power_limit_and_max_sm_clock"] = f"unavailable: {exc}"
    return info


def timed(fn, sets, reps=20):
    """average device ms per fn(*set): one pass over all sets captured in a CUDA graph, replayed `reps` times"""
    graph = torch.cuda.CUDAGraph()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for a in sets[:2]:                         # warm-up on the capture stream, results dropped at once
            fn(*a)
        side.synchronize()
        with torch.cuda.graph(graph, stream=side):
            keep = [fn(*a) for a in sets]
        graph.replay()
        side.synchronize()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record(side)
        for _ in range(reps):
            graph.replay()
        e.record(side)
        side.synchronize()
    del keep
    return s.elapsed_time(e) / (reps * len(sets))


def launches(fn, args):
    """(device activities of one eager call: kernels, memsets, copies; of those, libunetb200 launches)"""
    from torch.profiler import ProfilerActivity, profile
    fn(*args)
    torch.cuda.synchronize()
    n0 = ops.LAUNCHES
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn(*args)
        torch.cuda.synchronize()
    ours = ops.LAUNCHES - n0
    return sum(1 for ev in prof.events() if ev.device_type == torch.autograd.DeviceType.CUDA), ours


def criterion():
    g = torch.Generator().manual_seed(0)
    npix = B * S * S
    per_set = npix * (2 + 4)
    sets = []
    for _ in range(max(2, int(2 * L2_BYTES / per_set) + 1)):
        x = (torch.randn(B, 1, S, S, generator=g) * 3).to(dev).to(torch.bfloat16).requires_grad_(True)
        t = torch.randint(0, 2, (B, S, S), generator=g).to(dev).float()
        sets.append((x, t))

    def fused_pair(x, t):
        return torch.autograd.grad(UL.bce_dice_loss(x, t), x)[0]

    def fused(x, t):
        with torch.autocast("cuda", enabled=True):
            loss = UL.training_criterion(x, t)
        return torch.autograd.grad(loss, x)[0]

    def chain(x, t):
        with torch.autocast("cuda", enabled=True):
            p = x.squeeze(1)
            loss = F.binary_cross_entropy_with_logits(p, t)
            loss = loss + dice_loss(torch.sigmoid(p), t, multiclass=False)
            loss = loss + 0.25 * boundary_loss(p, t, edge_width=51, edge_weight=15)
        return torch.autograd.grad(loss, x)[0]

    # (no_grad: a live autograd graph would keep x's AccumulateGrad node on the default stream, which breaks the
    # captures below with cudaErrorStreamCaptureImplicit)
    with torch.no_grad(), torch.autocast("cuda", enabled=True):
        a = UL.training_criterion(*sets[0])
        p = sets[0][0].squeeze(1)
        b = (F.binary_cross_entropy_with_logits(p, sets[0][1]) + dice_loss(torch.sigmoid(p), sets[0][1])
             + 0.25 * boundary_loss(p, sets[0][1], edge_width=51, edge_weight=15))
    agree = abs(float(a) - float(b)) / abs(float(b))
    out = {"workload": f"B={B} {S}x{S}, bf16 logits [B,1,H,W], fp32 targets, forward + backward, "
                       f"{len(sets)} rotating input sets ({len(sets) * per_set / 1e6:.0f} MB) per graph pass",
           "fused_vs_chain_loss_rel": agree}
    arms = (("bce_dice_pair", fused_pair, 14), ("fused_criterion", fused, 20), ("reference_chain", chain, 20))
    for name, fn, bpp in arms:
        ms = timed(fn, sets)
        n_dev, n_ours = launches(fn, sets[0])
        out[name] = {"ms": ms, "device_activities": n_dev, "libunetb200_launches": n_ours,
                     "algorithmic_bytes": bpp * npix, "gbs": bpp * npix / ms / 1e6,
                     "frac_of_copy_peak": bpp * npix / ms / 1e6 / PEAK}
    out["chain_over_fused"] = out["reference_chain"]["ms"] / out["fused_criterion"]["ms"]
    return out


def train_steps(reps=30, rounds=2):
    torch.manual_seed(0)
    img = torch.rand(B, 1, S, S, device=dev).contiguous(memory_format=torch.channels_last)
    msk = torch.randint(0, 2, (B, S, S), device=dev)
    steps = {}
    for cls in ("UNet", "UNet_S"):
        for ncls in (1, 2):
            model = getattr(UM, cls)(1, ncls).to(dev).to(memory_format=torch.channels_last).train()
            opt = FusedRMSprop(model.parameters(), lr=1e-5, weight_decay=1e-8, momentum=0.999)

            def step(x, t, model=model, opt=opt, ncls=ncls):
                opt.zero_grad(set_to_none=True)
                with torch.autocast("cuda", enabled=True):
                    logits = model(x)
                    if ncls == 1:
                        loss = UL.training_criterion(logits, t)
                    else:
                        loss = UL.training_criterion(logits, t, boundary_coeff=0.2, edge_width=51, edge_weight=7)
                loss.backward()
                opt.step(clip_max_norm=1.0)
                return loss
            steps[f"{cls}(1,{ncls})"] = GraphedStep(step, (img, msk), warmup=2)
    res = {k: [] for k in steps}
    for _ in range(rounds):
        for k, g in steps.items():
            for _ in range(3):
                g.replay()
            torch.cuda.synchronize()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            for _ in range(reps):
                g.replay()
            e.record()
            torch.cuda.synchronize()
            ms = s.elapsed_time(e) / reps
            res[k].append({"ms_per_step": ms, "img_per_s": B * 1e3 / ms})
    loss_finite = {k: bool(torch.isfinite(g.static_loss).item()) for k, g in steps.items()}
    out = {"workload": f"B={B} {S}x{S}, bf16 autocast, whole-step CUDA graph, FusedRMSprop + clip 1.0, "
                       f"{reps} replays per round, {rounds} interleaved rounds",
           "steps": res, "loss_finite": loss_finite}
    for cls in ("UNet", "UNet_S"):
        best = {n: max(r["img_per_s"] for r in res[f"{cls}(1,{n})"]) for n in (1, 2)}
        out[f"{cls}_binary_over_2class"] = best[1] / best[2]
    return out


def main():
    assert torch.cuda.is_available(), "tools/bench_binary.py measures on a CUDA device"
    torch.cuda.set_device(dev)
    line = gpu_info()
    line["criterion"] = criterion()
    line["train_step"] = train_steps()
    print(json.dumps(line))


if __name__ == "__main__":
    main()
