#!/usr/bin/env python
"""bench.py -- the UNet hot path on N B200s, one line of JSON per run (rank 0).

    python bench.py --gpus 1 --steps K --warmup W                       # C2: BASELINE.json configs[1] (default)
    python bench.py --bilinear --precision tf32x3                        # C3: configs[2], fp32/TF32 exactness mode
    python bench.py --workload infer                                     # C5: configs[4], predict.py-style inference
    python bench.py --impl reference --gpus N --steps K ...              # reference arm: its CPU fp32 path
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...   # N > 1 (C4 = configs[3])
    python bench.py ... --dump-outputs DIR                               # + the last timed step's outputs as .npy

train: one step = forward + loss (CE + dice + 0.2*boundary_loss, the train.py:137-147 form) + backward (+ NCCL
gradient all-reduce when N > 1) + clip_grad_norm_ + RMSprop step (train.py:80,153-159) on 16 synthetic 1x512x512
images per GPU.  infer: one step = UNet(3,4).eval() forward under autocast + the predict.py:26-27 tail (bilinear
resize to the original size + argmax) on 8 synthetic 3x1024x1024 images per GPU; N > 1 = independent replicas.

Baselines printed beside the number (never the thing measured): ``cpu_baseline`` -- the reference's CPU fp32 path on
the box's host cores (the unmodified reference modules from the git-ignored baseline/_ref copy when it travelled
with the snapshot, else the oracle port); ``torch_gpu_baseline`` -- the same reference modules on the same GPU
through stock PyTorch (cuDNN / ATen, bf16 autocast, channels_last), i.e. what the reference runs on a B200 today.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "unet-medical-image-contour-segmentation_b200")
REF_DIR = os.path.join(ROOT, "baseline", "_ref")
for _p in (PKG, ROOT):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import torch  # noqa: E402

UNIT = "img/s"
# algorithmic conv FLOPs per image (SURVEY.md section 8d / BASELINE.md section 4): UNet(1,2,bilinear) fwd+bwd at 512x512,
# UNet(3,4,False) forward at 1024x1024
GFLOP_PER_IMG = {("train", False, 512): 1154.004, ("train", True, 512): 957.509, ("infer", False, 1024): 1541.759}
DTYPE_NAME = {"bf16": "bf16", "tf32": "tf32", "tf32x3": "tf32x3", "fp32": "f32"}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="train", choices=["train", "infer"])
    ap.add_argument("--precision", default="bf16", choices=["bf16", "tf32", "tf32x3", "fp32"],
                    help="bf16: autocast (configs[1]); tf32 / tf32x3 / fp32: autocast off, the fp32/TF32 exactness mode "
                         "(configs[2]) on tcgen05 kind::tf32, its 3-term split, or exact CUDA-core FMAs")
    ap.add_argument("--batch", type=int, default=None, help="images per GPU (default 16 train, 8 infer)")
    ap.add_argument("--size", type=int, default=None, help="default 512 train, 1024 infer")
    ap.add_argument("--bilinear", action="store_true")
    ap.add_argument("--model", default="UNet", choices=["UNet", "UNet_S", "UNet_T", "UNet_SA"],
                    help="UNet = BASELINE.json's model (the metric); the width variants of unet_model.py:52-189 (UNet_S is "
                         "what train.py:253 builds) run the same step for comparison, off the BASELINE metric")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-torch-baseline", action="store_true")
    ap.add_argument("--no-profile", action="store_true")
    ap.add_argument("--per-layer", action="store_true", help="add a per-layer conv table (`layers`) to the JSON line")
    ap.add_argument("--torch-optim", action="store_true",
                    help="torch.optim.RMSprop + clip_grad_norm_ instead of the fused multi-tensor kernels (A/B)")
    ap.add_argument("--graph", default="auto", choices=["auto", "on", "off"],
                    help="replay the whole step as one CUDA graph (auto: try, fall back to eager launches)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step returned as DIR/<name>.npy (float32; "
                         "at most 64 MB in all, larger arrays as a fixed seeded sample) to compare two builds")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.batch is None:
        a.batch = 16 if a.workload == "train" else 8
    if a.size is None:
        a.size = 512 if a.workload == "train" else 1024
    a.nc, a.ncls = (1, 2) if a.workload == "train" else (3, 4)
    return a


def metric_name(a):
    return f"{a.model.lower()}{a.size}_{'train' if a.workload == 'train' else 'infer'}_images_per_sec"


def model_class(pkg, a):
    """`UNet` from the package itself, the width variants from its unet_model module (the reference's __init__ exports
    UNet only)."""
    if a.model == "UNet":
        return pkg.UNet
    mod = sys.modules.get(pkg.__name__ + ".unet_model")
    if mod is None:
        import importlib
        mod = importlib.import_module(pkg.__name__ + ".unet_model")
    return getattr(mod, a.model)


def workload_text(a, per_gpu=True):
    if a.workload == "train":
        which = (f"BASELINE.json {'configs[2]' if a.bilinear else 'configs[1]; configs[3] when n_gpus > 1'}" if a.model == "UNet"
                 else "width variant of unet_model.py:52-189, same step as configs[1], off the BASELINE metric")
        return (f"{a.model}(1,2,bilinear={a.bilinear}) {a.precision} training step, batch {a.batch}/GPU, {a.size}x{a.size}, "
                f"CE+dice+0.2*boundary_loss(51,7), clip_grad_norm, RMSprop ({which})")
    which = "BASELINE.json configs[4]" if a.model == "UNet" else "width variant, off the BASELINE metric"
    return (f"{a.model}(3,4,bilinear={a.bilinear}).eval() {a.precision} predict.py-style inference (forward + resize + argmax), "
            f"batch {a.batch}/GPU, {a.size}x{a.size} ({which}; replicas when n_gpus > 1)")


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            with open(path) as f:
                d = json.load(f)
            return dict(hbm_gbs=float(d["hbm_gbs"]), tflops_burst=float(d["bf16_tflops"]),
                        tflops_sustained=float(d.get("bf16_tflops_sustained", d["bf16_tflops"])), source="measured")
        except Exception:  # noqa: BLE001
            pass
    return dict(hbm_gbs=6650.0, tflops_burst=1590.0, tflops_sustained=1400.0, source="fallback")


DUMP_BYTES = 64 << 20          # --dump-outputs writes at most this much


def step_outputs(a, result, params, buffers):
    """What a caller of one step receives.  train: the loss, and the parameters, gradients and floating-point
    buffers (BatchNorm running statistics) the step left behind, each flattened and concatenated in module order;
    infer: the label map."""
    if a.workload == "infer":
        return {"labels": result}

    def flat(ts):
        return torch.cat([t.detach().float().reshape(-1) for t in ts])
    return {"loss": result.detach().reshape(1), "params": flat(params),
            "grads": flat(p.grad for p in params),
            "buffers": flat(b for b in buffers if b.is_floating_point())}


def dump_outputs(path, arrays):
    """DIR/<name>.npy per array, float64 data as float64 and everything else as float32.  An array larger than an
    even share of DUMP_BYTES is replaced by a sample of its flattened elements at fixed, seeded indices (the same for
    every run with the same arguments)."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    share = DUMP_BYTES // len(arrays)
    for name, t in arrays.items():
        t = t.detach()
        t = t.double() if t.dtype == torch.float64 else t.float()
        cap = share // t.element_size()
        if t.numel() > cap:
            idx = torch.randperm(t.numel(), generator=torch.Generator().manual_seed(0))[:cap].sort().values
            t = t.reshape(-1)[idx.to(t.device)]
        np.save(os.path.join(path, f"{name}.npy"), t.cpu().numpy())


# ------------------------------------------------------------------------------------------------
# baselines: the reference's own modules (baseline/_ref, unmodified) or the oracle port
# ------------------------------------------------------------------------------------------------
def load_reference_modules():
    """The unmodified reference's ``unet``, ``utils.dice_score`` and ``utils.boundary_loss`` from the git-ignored
    baseline/_ref copy, imported under private names (they must not shadow the drop-in packages).  None if the copy
    did not travel with this snapshot."""
    if not os.path.isfile(os.path.join(REF_DIR, "unet", "unet_model.py")):
        return None
    import importlib.util

    def load(name, path, pkg_path=None):
        if name in sys.modules:
            return sys.modules[name]
        spec = importlib.util.spec_from_file_location(name, path, submodule_search_locations=pkg_path)
        mod = importlib.util.module_from_spec(spec)
        sys.modules[name] = mod
        spec.loader.exec_module(mod)
        return mod
    unet = load("_refunet", os.path.join(REF_DIR, "unet", "__init__.py"), [os.path.join(REF_DIR, "unet")])
    dice = load("_refdice", os.path.join(REF_DIR, "utils", "dice_score.py"))
    bnd = load("_refboundary", os.path.join(REF_DIR, "utils", "boundary_loss.py"))
    return unet, dice, bnd


def synthetic(a, rank, batch=None):
    B = a.batch if batch is None else batch
    gi = torch.Generator().manual_seed(1 + 1000 * rank)
    gm = torch.Generator().manual_seed(2 + 1000 * rank)
    img = torch.rand(B, a.nc, a.size, a.size, generator=gi)
    msk = torch.randint(0, a.ncls, (B, a.size, a.size), generator=gm, dtype=torch.long)
    return img, msk


class ReferenceStep:
    """train.py:113-159 (one optimisation step) / predict.py:15-29 (one predict_img call on a batch), restated around
    the reference's own modules -- train.py itself does not import as shipped (train.py:16,18).  device = cpu (fp32,
    amp off: the CPU baseline) or cuda (bf16 autocast, channels_last: what the reference runs on a GPU)."""

    def __init__(self, a, device, amp):
        import torch.nn.functional as F
        self.a, self.dev, self.amp, self.F = a, torch.device(device), amp, F
        mods = load_reference_modules()
        self.kind = "reference" if mods is not None else "port"
        torch.manual_seed(0)
        if mods is not None:
            refunet, self.dice, self.bnd = mods
            self.model = model_class(refunet, a)(a.nc, a.ncls, a.bilinear)
            self.dice_loss, self.boundary_loss = self.dice.dice_loss, self.bnd.boundary_loss
        else:
            if a.model != "UNet":
                raise RuntimeError("bench.py --model variants need the reference modules in baseline/_ref for their baseline legs")
            from oracle import unet_oracle as O           # the pinned restatement (baseline leg only)
            self.O = O
            self.state = O.build_state(a.nc, a.ncls, a.bilinear, seed=0)
            self.model = None
            self.dice_loss, self.boundary_loss = O.dice_loss, O.boundary_loss
        if self.model is not None:
            self.model = self.model.to(self.dev).to(memory_format=torch.channels_last)
            self.model.train() if a.workload == "train" else self.model.eval()
            params = list(self.model.parameters())
        else:
            self.names = self.O.param_names(self.state)
            self.state = {k: v.to(self.dev) for k, v in self.state.items()}
            params = [self.state[k].requires_grad_(True) for k in self.names]
        self.params = params
        if a.workload == "train":                        # train.py:80-84
            self.opt = torch.optim.RMSprop(params, lr=1e-5, weight_decay=1e-8, momentum=0.999, foreach=True)

    def forward(self, x):
        if self.model is not None:
            return self.model(x)
        return self.O.unet_forward(self.state, x, self.a.bilinear, training=(self.a.workload == "train"))

    def train_step(self, img, msk):
        F, a = self.F, self.a
        x = img.to(device=self.dev, dtype=torch.float32, memory_format=torch.channels_last)
        t = msk.to(device=self.dev, dtype=torch.long)
        with torch.autocast(self.dev.type, dtype=torch.bfloat16, enabled=self.amp):
            logits = self.forward(x)
            loss = F.cross_entropy(logits, t)
            loss = loss + self.dice_loss(F.softmax(logits, dim=1).float(),
                                         F.one_hot(t, a.ncls).permute(0, 3, 1, 2).float(), multiclass=True)
            loss = loss + 0.2 * self.boundary_loss(logits, t.float(), edge_width=51, edge_weight=7)
        self.opt.zero_grad(set_to_none=True)
        loss.backward()
        torch.nn.utils.clip_grad_norm_(self.params, 1.0)
        self.opt.step()
        return loss

    def infer_step(self, img):
        F = self.F
        x = img.to(device=self.dev, dtype=torch.float32, memory_format=torch.channels_last)
        with torch.no_grad(), torch.autocast(self.dev.type, dtype=torch.bfloat16, enabled=self.amp):
            out = self.forward(x)
            out = F.interpolate(out, (x.shape[2], x.shape[3]), mode="bilinear")
            return out.argmax(dim=1)

    def step(self, img, msk):
        return self.train_step(img, msk) if self.a.workload == "train" else self.infer_step(img)

    def buffers(self):
        if self.model is not None:
            return list(self.model.buffers())
        return [v for k, v in self.state.items() if k not in self.names]


def cpu_reference_rate(a, steps, warmup, budget_s, batch, dump=None):
    """img/s of the reference's CPU fp32 step, all host threads; `batch` images per step (a bounded sample of the
    workload), at most `budget_s` seconds, at least one timed step.  `dump`: a directory for the outputs of the last
    timed step (--dump-outputs)."""
    torch.set_num_threads(os.cpu_count() or 1)
    ref = ReferenceStep(a, "cpu", amp=False)
    img, msk = synthetic(a, 0, batch)
    times, done_warm = [], 0
    t_start = time.perf_counter()
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        out = ref.step(img, msk)
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
        else:
            done_warm += 1
        elapsed = time.perf_counter() - t_start
        if times and elapsed + dt > budget_s:
            break
        if not times and done_warm >= 1 and elapsed + 2 * dt > budget_s:
            warmup = done_warm                   # cut the warm-up short: keep at least one timed step
    if not times:
        times = [dt]
    if dump:
        dump_outputs(dump, step_outputs(a, out, ref.params, ref.buffers()))
    med = statistics.median(times)
    return batch / med, len(times), done_warm, med, ref.kind


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # one timed step = a bounded sample of the workload: 2 images.  Measured on the 16 host cores of a B200 machine
    # (profiles/r2_bench_reference_b16.json): 2 images take 1.44 s/step (1.39 img/s), but the full batch of 16 took
    # 596 s for ONE step (0.027 img/s: the fp32 activations + autograd state of B=16 at 512x512 no longer fit the
    # host's memory comfortably), so the full batch would neither finish a run of 20 steps nor flatter the CPU.
    # --steps sets the number of timed steps exactly: no time budget here.
    batch = min(a.batch, 2)
    rate, n, nw, med, kind = cpu_reference_rate(a, a.steps, min(a.warmup, 1), budget_s=float("inf"), batch=batch,
                                                dump=a.dump_outputs)
    cores = os.cpu_count() or 1
    src = ("unmodified reference modules (baseline/_ref: unet, utils.dice_score, utils.boundary_loss)" if kind == "reference"
           else "oracle port of the reference step (torch-CPU fp32 restatement; baseline/_ref did not travel)")
    sample = (f"{src}, CPU fp32, {cores} threads, {batch} images per step of the {a.size}x{a.size} workload, "
              f"{nw} warm-up + {n} timed steps, median {med:.2f} s/step")
    line = {
        "impl": "reference", "metric": metric_name(a), "value": rate, "unit": UNIT, "n_gpus": a.gpus, "steps": n,
        "warmup": nw, "ms_per_step": med * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_text(a), "per_step_sample": f"{batch} images"},
        "cpu_baseline": {"value": rate, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def torch_gpu_baseline(a, dev, img_h, msk_h, steps=8, warmup=3):
    """The reference's modules through stock PyTorch on this GPU (cuDNN / ATen; bf16 autocast for the bf16 workloads,
    TF32 convs otherwise; channels_last; eager launches, as train.py / predict.py run them).  Informational."""
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.benchmark)
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = (a.precision != "fp32")
    torch.backends.cudnn.benchmark = True
    try:
        ref = ReferenceStep(a, dev, amp=(a.precision == "bf16"))
        x, t = img_h.to(dev), msk_h.to(dev)
        for _ in range(warmup):
            ref.step(x, t)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            ref.step(x, t)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        return {"value": a.batch / ms * 1e3, "unit": UNIT, "ms_per_step": ms, "steps": steps, "kind": ref.kind,
                "what": ("reference modules on stock PyTorch (cuDNN " + str(torch.backends.cudnn.version()) + "), "
                         + ("bf16 autocast" if a.precision == "bf16" else ("TF32" if a.precision != "fp32" else "fp32"))
                         + ", channels_last, eager, inputs resident in HBM, 1 GPU")}
    except Exception as exc:  # noqa: BLE001
        return {"unavailable": f"{type(exc).__name__}: {exc}"[:200]}
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.benchmark = old
        torch.cuda.empty_cache()


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(gpu_index), f"--query-gpu={self.Q}",
                                       "--format=csv,noheader,nounits", "-lms", "50"], stdout=self.f,
                                      stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.f.read().splitlines():
            parts = [s.strip() for s in ln.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
            except ValueError:
                continue
            for nm, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        self.f.close()
        os.unlink(self.f.name)
        if sm:
            s = sorted(sm)                       # "under load": drop the lowest quartile (ramp-up samples)
            out["sm_mhz"] = statistics.median(s[len(s) // 4:])
            out["sm_max_mhz"] = max(mx)
        out["reasons"] = sorted(reasons)
        out["samples"] = len(sm)
        return out


def roofline_tables(a, rec, peaks, nsteps):
    """Per-kernel-class table + the `roofline` objects from an instrumented pass (CUDA events around every C-ABI call,
    each call timed alone on its stream => the peak a class is held against is the BURST figure; the sustained one is
    given next to it).  A conv class whose arithmetic intensity (algorithmic FLOP / algorithmic byte) is below the
    ridge point is HBM-bound and is labelled and rated as such (the full-resolution ConvTranspose GEMMs)."""
    from unetb200 import ops
    per_layer = ops.summarize_profile(rec)
    summ = {}
    for name, d in per_layer.items():                     # class = name without the [M=..,N=..,K=..] tag
        cls = name.split("[")[0]
        e = summ.setdefault(cls, dict(ms=0.0, calls=0, flops=0.0, bytes=0.0))
        for k in e:
            e[k] += d[k]
    out = {}
    if a.per_layer:
        out["layers"] = {n: {"ms": d["ms"] / nsteps, "tflops": d["flops"] / (d["ms"] * 1e-3) / 1e12}
                         for n, d in sorted(per_layer.items(), key=lambda kv: -kv[1]["ms"]) if "[" in n}
    ridge = peaks["tflops_burst"] * 1e12 / (peaks["hbm_gbs"] * 1e9)
    tot_ms = sum(d["ms"] for d in summ.values()) or 1.0
    kernels = {}
    for name, d in sorted(summ.items(), key=lambda kv: -kv[1]["ms"]):
        ent = {"ms_per_step": d["ms"] / nsteps, "share": d["ms"] / tot_ms, "launches_per_step": d["calls"] // nsteps}
        sec = d["ms"] * 1e-3
        tensor = d["flops"] > 0 and (d["bytes"] <= 0 or d["flops"] / d["bytes"] >= ridge)
        if d["flops"] > 0:
            ent["tflops"] = d["flops"] / sec / 1e12
        if d["bytes"] > 0:
            ent["gbs"] = d["bytes"] / sec / 1e9
        if tensor:
            ent["bound"] = "tensor"
            ent["frac_of_peak"] = ent["tflops"] / peaks["tflops_burst"]
            ent["frac_of_sustained_peak"] = ent["tflops"] / peaks["tflops_sustained"]
        elif d["bytes"] > 0:
            ent["bound"] = "hbm"
            ent["frac_of_peak"] = ent["gbs"] / peaks["hbm_gbs"]
            if d["flops"] > 0:
                ent["flop_per_byte"] = d["flops"] / d["bytes"]
        kernels[name] = ent
    out["kernels"] = kernels
    if not kernels:
        return out
    dom = next(iter(kernels))
    kd, sd = kernels[dom], summ[dom]
    traffic, traffic_src = None, None
    try:                                  # DRAM bytes per launch of that kernel class from the committed ncu pass
        if a.model != "UNet" or a.workload != "train":
            raise LookupError("the committed ncu pass is of BASELINE configs[1]")
        import glob
        tj = sorted(glob.glob(os.path.join(ROOT, "profiles", "kernel_traffic_r*.json")))[-1]
        with open(tj) as f:
            tdata = json.load(f)
        ent_t = tdata["per_class"].get(dom)
        if ent_t is None and dom in ("conv_fprop_tc", "conv_dgrad_tc"):
            ent_t = tdata["per_class"].get("conv_fprop_tc+conv_dgrad_tc")
        if ent_t:
            traffic, traffic_src = ent_t["dram_bytes_per_launch"], os.path.basename(tj) + ": " + tdata["source"]
    except Exception:  # noqa: BLE001
        pass
    common = {"kernel": dom, "traffic": traffic, "traffic_unit": "DRAM bytes per launch (ncu)",
              "traffic_source": traffic_src, "launches": sd["calls"], "avg_launch_ms": sd["ms"] / sd["calls"]}
    if kd.get("bound") == "tensor":
        out["roofline"] = {"bound": "tensor", "achieved": kd["tflops"], "peak": peaks["tflops_burst"], "unit": "TFLOP/s",
                           "frac": kd["frac_of_peak"], "peak_sustained": peaks["tflops_sustained"],
                           "frac_of_sustained": kd["frac_of_sustained_peak"],
                           "algorithmic_flops_per_launch": sd["flops"] / sd["calls"],
                           "peak_source": peaks["source"] + " (bf16 cuBLAS burst; each launch is event-timed alone)",
                           **common}
    else:
        out["roofline"] = {"bound": "hbm", "achieved": kd.get("gbs"), "peak": peaks["hbm_gbs"], "unit": "GB/s",
                           "frac": kd.get("frac_of_peak"), "algorithmic_bytes_per_launch": sd["bytes"] / sd["calls"],
                           "peak_source": peaks["source"] + " (copy)", **common}
    hbm = [(n, k) for n, k in kernels.items() if k.get("bound") == "hbm"]
    if hbm:
        hn, hk = hbm[0]
        out["roofline_hbm"] = {"bound": "hbm", "kernel": hn, "achieved": hk["gbs"], "peak": peaks["hbm_gbs"],
                               "unit": "GB/s", "frac": hk["frac_of_peak"], "peak_source": peaks["source"] + " (copy)",
                               "launches": summ[hn]["calls"], "avg_launch_ms": summ[hn]["ms"] / summ[hn]["calls"]}
    conv = [(n, d) for n, d in summ.items() if n.startswith("conv_")]
    conv_ms = sum(d["ms"] for _, d in conv) / nsteps
    conv_fl = sum(d["flops"] for _, d in conv) / nsteps
    if conv_ms > 0:
        tf = conv_fl / (conv_ms * 1e-3) / 1e12
        out["conv_tensor_util"] = {"tflops": tf, "frac_of_burst_peak": tf / peaks["tflops_burst"],
                                   "frac_of_sustained_peak": tf / peaks["tflops_sustained"], "conv_ms_per_step": conv_ms}
    mem_ms = sum(d["ms"] for n, d in summ.items() if kernels[n].get("bound") != "tensor") / nsteps
    out["memory_bound_ms_per_step"] = mem_ms
    return out


def set_precision(a):
    """bf16 -> autocast on.  Otherwise autocast off and the library's fp32 policy (functional.conv_algo)."""
    if a.precision != "bf16":
        os.environ["UNET_B200_PRECISION"] = a.precision
    return a.precision == "bf16"


def run_ours(a):
    import torch.distributed as dist
    import unet
    from unetb200 import ddp, ops

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the UNet hot path has no CPU fallback (use --impl reference for "
                         "the CPU arm)")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev, timeout=__import__("datetime").timedelta(seconds=180))
    ctx = dict(a=a, world=world, rank=rank, local=local, dev=dev, dist=dist, unet=unet, ddp=ddp, ops=ops,
               amp=set_precision(a))
    line = (bench_train if a.workload == "train" else bench_infer)(ctx)
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def _sync_all(ctx):
    torch.cuda.synchronize()
    if ctx["world"] > 1:
        ctx["dist"].barrier()
        torch.cuda.synchronize()


def _timed(ctx, fn, n):
    """n calls of fn bracketed by barrier + synchronize on both sides, CUDA events, max over ranks (ms)."""
    _sync_all(ctx)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    _sync_all(ctx)
    ms = e0.elapsed_time(e1)
    if ctx["world"] > 1:
        t = torch.tensor([ms], device=ctx["dev"])
        ctx["dist"].all_reduce(t, op=ctx["dist"].ReduceOp.MAX)
        ms = t.item()
    return ms


def _base_line(ctx, ms, ms_e2e, launches, clocks, h2d, d2h):
    a, world = ctx["a"], ctx["world"]
    total = a.batch * world * a.steps
    return {
        "metric": metric_name(a), "value": total / (ms / 1e3), "unit": UNIT, "n_gpus": world, "steps": a.steps,
        "warmup": a.warmup, "ms_per_step": ms / a.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": DTYPE_NAME[a.precision], "data": "synthetic",
        "config": {"workload": workload_text(a), "global_batch": a.batch * world,
                   "parallelism": f"dp{world}" if a.workload == "train" else f"replicas{world}",
                   "l2": "activations per step (~10 GB) far exceed the 126 MB L2; no flush needed", "random_init": True},
        "e2e": {"value": total / (ms_e2e / 1e3), "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": ms_e2e / a.steps},
        "gpu_launches": launches, "clocks": clocks,
    }


def _add_baselines(ctx, line, img_h, msk_h):
    a = ctx["a"]
    if ctx["rank"] != 0 or ctx["world"] != 1:
        return
    if not a.no_torch_baseline:
        line["torch_gpu_baseline"] = torch_gpu_baseline(a, ctx["dev"], img_h, msk_h)
    if not a.no_cpu_baseline:
        batch = 2 if a.workload == "train" else 1
        rate, n, nw, med, kind = cpu_reference_rate(a, steps=3, warmup=1, budget_s=40.0, batch=batch)
        line["cpu_baseline"] = {"value": rate, "unit": UNIT, "cores": os.cpu_count() or 1, "kind": kind,
                                "sample": f"{'unmodified reference modules (baseline/_ref)' if kind == 'reference' else 'oracle port'}"
                                          f", CPU fp32, same step on {batch} images of {a.size}x{a.size}, "
                                          f"{nw} warm-up + {n} timed, median {med:.2f} s/step"}


def bench_train(ctx):
    a, world, rank, dev, dist, ddp, ops = (ctx[k] for k in ("a", "world", "rank", "dev", "dist", "ddp", "ops"))
    from unetb200 import losses as UL
    B, S, amp = a.batch, a.size, ctx["amp"]
    torch.manual_seed(0)
    model = model_class(ctx["unet"], a)(1, 2, a.bilinear).to(dev).to(memory_format=torch.channels_last).train()
    if world > 1:
        ddp.broadcast_module_state(model)
    bucket_mb = int(os.environ.get("UNETB200_DDP_BUCKET_MB", "32"))
    reducer = ddp.GradAllReducer(model, bucket_bytes=bucket_mb << 20) if world > 1 else None
    if a.torch_optim:
        opt = torch.optim.RMSprop(model.parameters(), lr=1e-5, weight_decay=1e-8, momentum=0.999, foreach=True,
                                  capturable=(a.graph != "off"))

        def clip_and_step():
            torch.nn.utils.clip_grad_norm_(model.parameters(), 1.0)
            opt.step()
    else:
        from unetb200.optim import FusedRMSprop      # same arithmetic (tests: optim group), two launches
        opt = FusedRMSprop(model.parameters(), lr=1e-5, weight_decay=1e-8, momentum=0.999)

        def clip_and_step():
            opt.step(clip_max_norm=1.0)

    img_h, msk_h = synthetic(a, rank)
    img_h, msk_h = img_h.pin_memory(), msk_h.pin_memory()
    img_d = img_h.to(dev).contiguous(memory_format=torch.channels_last)
    msk_d = msk_h.to(dev)

    def fwd_loss(x, t):
        with torch.autocast("cuda", enabled=amp):
            return UL.training_criterion(model(x), t, boundary_coeff=0.2, edge_width=51, edge_weight=7)

    def step(x, t):
        opt.zero_grad(set_to_none=True)
        loss = fwd_loss(x, t)
        loss.backward()
        if reducer is not None:
            reducer.finish()
        clip_and_step()
        return loss

    copy_stream = torch.cuda.Stream(device=dev)

    def prefetch():
        """H2D copy of one step's inputs from pinned host memory on the copy stream (a loader's prefetch)."""
        with torch.cuda.stream(copy_stream):
            x = img_h.to(device=dev, dtype=torch.float32, non_blocking=True, memory_format=torch.channels_last)
            t = msk_h.to(device=dev, dtype=torch.long, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(copy_stream)
        return x, t, ev

    def e2e_steps(n):
        """n end-to-end steps: every step's inputs cross PCIe inside the loop (the copy of step i+1 overlaps the
        compute of step i, as train.py's DataLoader(pin_memory=True) + non_blocking copies allow) and every
        step ends with the D2H read of its loss (train.py:163)."""
        nxt = prefetch()
        out = 0.0
        for i in range(n):
            x, t, ev = nxt
            torch.cuda.current_stream().wait_event(ev)
            x.record_stream(torch.cuda.current_stream())
            t.record_stream(torch.cuda.current_stream())
            loss = step(x, t)                 # asynchronous launch (graph replay)
            if i + 1 < n:
                nxt = prefetch()              # issued while the step runs: no host work between the loss read and the next launch
            out = loss.item()
        return out

    first_loss = None
    for _ in range(a.warmup):
        lw = step(img_d, msk_d)
        if first_loss is None:
            first_loss = float(lw.detach())
        del lw      # a live loss tensor keeps its autograd graph (and default-stream AccumulateGrad nodes) alive,
        #             which breaks the CUDA-graph capture below (cudaErrorStreamCaptureImplicit)
    _sync_all(ctx)
    # ---- whole-step CUDA graph (falls back to eager launches if capture is not possible) -------
    eager_step = step
    graphed, graph_note = None, "off"
    l0 = ops.LAUNCHES
    eager_step(img_d, msk_d)             # (result dropped at once, see above)
    launches_per_step = ops.LAUNCHES - l0
    seg = None
    if a.graph != "off":
        try:
            from unetb200.graph import GraphedStep
            if world == 1:
                graphed = GraphedStep(eager_step, (img_d, msk_d), warmup=2)
                graph_note = "on"
            else:
                # N > 1: the backward pass is captured as a few graph SEGMENTS; between two segments the buckets whose
                # gradients are complete are all-reduced eagerly on NCCL's stream while the next segment runs
                # (ddp.SegmentedStep) -- only the last, small bucket (inc.*) is exposed before the optimizer graph
                reducer.remove()
                for p in model.parameters():
                    p.grad = None
                seg = ddp.SegmentedStep(model, fwd_loss, clip_and_step, (img_d, msk_d))
                graphed = seg
                graph_note = seg.describe()
        except Exception as exc:  # noqa: BLE001
            if a.graph == "on":
                raise
            import traceback
            sys.stderr.write(f"[rank {rank}] CUDA graph capture failed:\n" + traceback.format_exc())
            graphed, seg, graph_note = None, None, f"capture failed, eager launches: {type(exc).__name__}: {exc}"[:200]
            if reducer is not None:
                reducer.remove()
                reducer = ddp.GradAllReducer(model, bucket_bytes=bucket_mb << 20)       # back to hook-driven eager mode
            torch.cuda.synchronize()
        if world > 1:                                     # every rank must take the same path
            flag = torch.tensor([1 if graphed is not None else 0], device=dev)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
            if flag.item() == 0 and graphed is not None:
                graphed = seg = None
                reducer.remove()
                reducer = ddp.GradAllReducer(model, bucket_bytes=bucket_mb << 20)
    if graphed is not None:
        def step(x, t):                                   # noqa: F811  (x, t are already in the static buffers when equal)
            if x is not graphed.static_inputs[0]:
                graphed.load(x, t)
            return graphed.replay()
        img_d, msk_d = graphed.static_inputs
        for _ in range(2):
            step(img_d, msk_d)
    _sync_all(ctx)
    sampler = ClockSampler(ctx["local"]) if rank == 0 else None
    last = [None]

    def timed_step():
        last[0] = step(img_d, msk_d)
    ms = _timed(ctx, timed_step, a.steps)
    clocks = sampler.stop() if sampler else {}
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, step_outputs(a, last[0], list(model.parameters()), list(model.buffers())))
    last[0] = None                  # a live loss keeps its autograd graph alive (see the warm-up above)
    e2e_steps(2)
    ms_e2e = _timed(ctx, lambda: e2e_steps(a.steps), 1)
    last_loss = float(step(img_d, msk_d).detach())
    torch.cuda.synchronize()

    line = _base_line(ctx, ms, ms_e2e, launches_per_step * a.steps, clocks,
                      img_h.numel() * 4 + msk_h.numel() * 8, 4)
    line["cuda_graph"] = graph_note
    line["first_loss"], line["final_loss"] = first_loss, last_loss
    # the step really trains: same synthetic batch every step, so the loss must not blow up (a scheduling bug
    # that feeds the optimizer stale gradients shows here)
    line["loss_sane"] = bool(first_loss is not None and last_loss == last_loss and last_loss < 1.2 * first_loss)
    peaks = measured_peaks()
    gf_img = GFLOP_PER_IMG.get(("train", a.bilinear, S)) if a.model == "UNet" else None
    if gf_img:
        conv_tf = gf_img * 1e9 * line["value"] / world / 1e12
        line["step_conv_tflops_per_gpu"] = conv_tf
        line["step_frac_of_bf16_peak"] = conv_tf / peaks["tflops_burst"]
        line["step_frac_of_bf16_sustained_peak"] = conv_tf / peaks["tflops_sustained"]

    # ---- per-kernel roofline: instrumented pass (CUDA events around every C-ABI call), eager launches ----------
    step = eager_step
    if seg is not None:
        seg.release()
        reducer = ddp.GradAllReducer(model, bucket_bytes=bucket_mb << 20)
    if world > 1 and not a.no_profile and rank != 0:
        for _ in range(2):                                # every rank takes part (the steps all-reduce); rank 0 records
            step(img_d, msk_d)
        torch.cuda.synchronize()
    if rank == 0 and not a.no_profile:
        os.environ["UNETB200_PROFILE_SHAPES"] = "1"
        with ops.profile() as rec:
            for _ in range(2):
                step(img_d, msk_d)
        torch.cuda.synchronize()
        os.environ.pop("UNETB200_PROFILE_SHAPES", None)
        line.update(roofline_tables(a, rec, peaks, 2))
    del graphed, seg
    _add_baselines(ctx, line, img_h, msk_h)
    return line


def bench_infer(ctx):
    """configs[4]: predict.py-style inference; with N > 1 every rank is an independent replica (no collective)."""
    a, world, rank, dev, ops = (ctx[k] for k in ("a", "world", "rank", "dev", "ops"))
    from unetb200 import eval_tail as UE
    B, S, amp = a.batch, a.size, ctx["amp"]
    torch.manual_seed(0)
    model = model_class(ctx["unet"], a)(a.nc, a.ncls, a.bilinear).to(dev).to(memory_format=torch.channels_last).eval()
    img_h, msk_h = synthetic(a, rank)
    img_h = img_h.pin_memory()
    img_d = img_h.to(dev).contiguous(memory_format=torch.channels_last)

    def step(x):
        with torch.inference_mode(), torch.autocast("cuda", enabled=amp):
            return UE.resize_argmax(model(x), (S, S))

    for _ in range(a.warmup):
        step(img_d)
    torch.cuda.synchronize()
    l0 = ops.LAUNCHES
    step(img_d)
    launches_per_step = ops.LAUNCHES - l0
    graph_note, replay = "off", None
    if a.graph != "off":
        try:
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, capture_error_mode="thread_local"):
                static_out = step(img_d)
            replay, graph_note = g.replay, "on"
        except Exception as exc:  # noqa: BLE001
            if a.graph == "on":
                raise
            graph_note = f"capture failed, eager launches: {type(exc).__name__}: {exc}"[:200]
            torch.cuda.synchronize()
    run = replay if replay is not None else (lambda: step(img_d))
    for _ in range(2):
        run()
    _sync_all(ctx)
    sampler = ClockSampler(ctx["local"]) if rank == 0 else None
    last = [None]

    def timed_step():
        last[0] = run()
    ms = _timed(ctx, timed_step, a.steps)
    clocks = sampler.stop() if sampler else {}
    if a.dump_outputs and rank == 0:             # a graph replay returns nothing: its label map is static_out
        dump_outputs(a.dump_outputs, step_outputs(a, static_out if replay is not None else last[0], None, None))

    # end to end through the reference-facing call: predict_img(model, host images, device) -> label map on the host
    copy_stream = torch.cuda.Stream(device=dev)
    d2h_stream = torch.cuda.Stream(device=dev)
    out_h = torch.empty((B, S, S), dtype=torch.int64).pin_memory()

    def e2e_steps(n):
        def prefetch():
            with torch.cuda.stream(copy_stream):
                x = img_h.to(device=dev, non_blocking=True, memory_format=torch.channels_last)
                ev = torch.cuda.Event()
                ev.record(copy_stream)
            return x, ev
        nxt = prefetch()
        cur = torch.cuda.current_stream()
        for i in range(n):
            x, ev = nxt
            cur.wait_event(ev)
            x.record_stream(cur)
            labels = UE.predict_img(model, x, dev)        # asynchronous launches
            if i + 1 < n:
                nxt = prefetch()
            # the label map goes back to the host on its own stream, so the device -> host copy of step i overlaps the
            # compute of step i + 1 (on boxes with a slow PCIe path the in-stream copy cost 2.7 ms of a 10.4 ms step)
            done = torch.cuda.Event()
            done.record(cur)
            with torch.cuda.stream(d2h_stream):
                d2h_stream.wait_event(done)
                out_h.copy_(labels, non_blocking=True)
                labels.record_stream(d2h_stream)
        d2h_stream.synchronize()
        cur.synchronize()

    e2e_steps(2)
    ms_e2e = _timed(ctx, lambda: e2e_steps(a.steps), 1)
    line = _base_line(ctx, ms, ms_e2e, launches_per_step * a.steps, clocks, img_h.numel() * 4, out_h.numel() * 8)
    line["cuda_graph"] = graph_note
    peaks = measured_peaks()
    gf_img = GFLOP_PER_IMG.get(("infer", a.bilinear, S)) if a.model == "UNet" else None
    if gf_img and a.nc == 3 and a.ncls == 4:
        conv_tf = gf_img * 1e9 * line["value"] / world / 1e12
        line["step_conv_tflops_per_gpu"] = conv_tf
        line["step_frac_of_bf16_peak"] = conv_tf / peaks["tflops_burst"]
    if rank == 0 and not a.no_profile:
        os.environ["UNETB200_PROFILE_SHAPES"] = "1"
        with ops.profile() as rec:
            for _ in range(2):
                step(img_d)
        torch.cuda.synchronize()
        os.environ.pop("UNETB200_PROFILE_SHAPES", None)
        line.update(roofline_tables(a, rec, peaks, 2))
    _add_baselines(ctx, line, img_h, msk_h)
    return line


def main():
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)


if __name__ == "__main__":
    main()
