"""Cost of synchronised BatchNorm (nn.SyncBatchNorm.convert_sync_batchnorm(UNet)) on the data-parallel training step.

    python -m torch.distributed.run --nproc-per-node N tools/bench_syncbn.py [--out FILE] [--rounds R] [--steps K]

Within one run, per configuration, it alternates per-replica BatchNorm and SyncBatchNorm R times, both driven by
ddp.SegmentedStep (graph-replayed step with bucketed NCCL all-reduces between backward segments), K timed steps each,
CUDA-event timed on rank 0 after a device synchronise of every rank:
  C2     16 images / GPU at 512^2, bf16 autocast (BASELINE.json configs[1] per GPU)
  small   2 images / GPU at 1024^2 (few images per GPU: where synchronised statistics matter)
It also times the exchange kernel alone (unetb200_bn_sync_finalize, ~2000 back-to-back calls, CUDA events) at C = 64
and C = 1024.  Rank 0 writes one JSON object (to FILE, or stdout) with the GPU name and power limit.
"""
import argparse
import json
import os
import subprocess
import sys

import torch
import torch.distributed as dist
import torch.nn as nn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (os.path.join(ROOT, "unet-medical-image-contour-segmentation_b200"), ROOT):
    if p not in sys.path:
        sys.path.insert(0, p)

import unet  # noqa: E402
from unetb200 import ddp, ops  # noqa: E402
from unetb200 import losses as UL  # noqa: E402
from unetb200.optim import FusedRMSprop  # noqa: E402

CONFIGS = {"C2": (16, 512), "small": (2, 1024)}


def gpu_info(dev):
    info = {"gpu": torch.cuda.get_device_name(dev)}
    try:
        out = subprocess.check_output(["nvidia-smi", "-i", str(dev.index), "--query-gpu=power.limit,clocks.max.sm",
                                       "--format=csv,noheader"], text=True, timeout=30).strip()
        info["power_limit_and_max_sm_clock"] = out
    except (OSError, subprocess.SubprocessError) as exc:
        info["power_limit_and_max_sm_clock"] = f"unavailable: {exc}"
    return info


def make_step(sync, B, S, rank, dev):
    torch.manual_seed(0)
    model = unet.UNet(1, 2)
    if sync:
        model = nn.SyncBatchNorm.convert_sync_batchnorm(model)
    model = model.to(dev).to(memory_format=torch.channels_last).train()
    ddp.broadcast_module_state(model)
    opt = FusedRMSprop(model.parameters(), lr=1e-5, weight_decay=1e-8, momentum=0.999)
    g = torch.Generator().manual_seed(1 + rank)
    x = torch.rand(B, 1, S, S, generator=g).to(dev).contiguous(memory_format=torch.channels_last)
    t = torch.randint(0, 2, (B, S, S), generator=g).to(dev)

    def fwd_loss(xx, tt):
        with torch.autocast("cuda"):
            return UL.training_criterion(model(xx), tt, boundary_coeff=0.2, edge_width=51, edge_weight=7)

    step = ddp.SegmentedStep(model, fwd_loss, lambda: opt.step(clip_max_norm=1.0), (x, t))
    return step


def time_steps(step, n):
    torch.cuda.synchronize()
    dist.barrier()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(n):
        step.replay()
    e.record()
    torch.cuda.synchronize()
    ms = torch.tensor([s.elapsed_time(e) / n], device=step.static_loss.device)
    dist.all_reduce(ms, op=dist.ReduceOp.MAX)          # the step of the slowest rank
    return float(ms)


def time_exchange(dev, Cc, n):
    pg = ddp.bn_sync_group(nn.SyncBatchNorm(Cc), dev)
    stats = torch.rand(2 * Cc, dtype=torch.float64, device=dev) + 1.0
    gamma, beta = torch.ones(Cc, device=dev), torch.zeros(Cc, device=dev)
    for _ in range(20):
        ops.bn_sync_finalize(pg, stats, 4096, gamma, beta, 1e-5, 0.0, None, None, Cc)
    # the calls are captured in one graph (one launch each on replay) so host time does not hide the kernel time
    g = torch.cuda.CUDAGraph()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        with torch.cuda.graph(g):
            for _ in range(n):
                ops.bn_sync_finalize(pg, stats, 4096, gamma, beta, 1e-5, 0.0, None, None, Cc)
    torch.cuda.current_stream().wait_stream(side)
    g.replay()
    torch.cuda.synchronize()
    dist.barrier()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    g.replay()
    e.record()
    torch.cuda.synchronize()
    us = torch.tensor([s.elapsed_time(e) * 1e3 / n], device=dev)
    dist.all_reduce(us, op=dist.ReduceOp.MAX)
    return float(us)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--configs", default="C2,small")
    ap.add_argument("--exchange-calls", type=int, default=2000)
    a = ap.parse_args()
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", device_id=dev)
    res = {"world": world, **gpu_info(dev), "configs": {}, "exchange_us": {}}
    for name in a.configs.split(","):
        B, S = CONFIGS[name]
        ms = {"per_replica": [], "sync": []}
        for _ in range(a.rounds):
            for kind in ("per_replica", "sync"):
                step = make_step(kind == "sync", B, S, rank, dev)
                ms[kind].append(time_steps(step, a.steps))
                step.release()
                del step
                torch.cuda.empty_cache()
        med = {k: sorted(v)[len(v) // 2] for k, v in ms.items()}
        res["configs"][name] = {
            "images_per_gpu": B, "size": S, "step_ms": ms, "median_step_ms": med,
            "img_per_s": {k: world * B * 1e3 / v for k, v in med.items()},
            "sync_over_per_replica_img_per_s": med["per_replica"] / med["sync"]}
    for Cc in (64, 1024):
        res["exchange_us"][str(Cc)] = time_exchange(dev, Cc, a.exchange_calls)
    res["exchange_calls"] = a.exchange_calls
    ddp.destroy_peer_groups()
    if rank == 0:
        text = json.dumps(res, indent=1)
        if a.out:
            os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
            with open(a.out, "w") as f:
                f.write(text + "\n")
        print(text, flush=True)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
