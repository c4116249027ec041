"""GPU parity checks (through the C ABI) of the callers either side of the step: the uint8 input pipeline
(unetb200.data) and the evaluate / predict tails (unetb200.eval_tail), against oracle/io_oracle.py and the
fixtures generated from the reference (tests/golden/golden_io_v1.pt).  Byte / index work: the bar is bit-exact
(err = number of differing elements, tol = 0); the dice scalar is compared at 1e-6.

Each check returns a list of (label, error, tolerance), like tests/gpu_checks.py."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "unet-medical-image-contour-segmentation_b200")
for _p in (PKG, ROOT):
    if _p not in sys.path:
        sys.path.insert(0, _p)

from oracle import io_oracle as IO  # noqa: E402
from unetb200 import data as UD  # noqa: E402
from unetb200 import eval_tail as UE  # noqa: E402

DEV = "cuda"


def load_golden_io():
    """The label maps (`out_msk`, `idx`) are stored as uint8 to keep the file small; they are int64 in the reference
    and are widened back here."""
    g = torch.load(os.path.join(ROOT, "tests", "golden", "golden_io_v1.pt"), weights_only=False)
    for cases in g.values():
        for c in cases:
            for k in ("out_msk", "idx"):
                if k in c:
                    c[k] = c[k].long()
    return g


def ndiff(a, b):
    a, b = a.detach().cpu(), b.detach().cpu()
    if a.shape != b.shape or a.dtype != b.dtype:
        return float("inf")
    return float((a != b).sum().item())


def check_pipeline(gio=None):
    gio = gio or load_golden_io()
    out = []
    # reference fixtures, one sample at a time (every rotation, gray / RGB / the unscaled 0-1 image)
    for c in gio["pipeline"]:
        r = UD.preprocess_batch([c["img"].numpy()], [c["msk"].numpy()], [c["k"]], device=DEV)
        out.append((f"pipe_img_{c['tag']}_k{c['k']}", ndiff(r["image"][0], c["out_img"]), 0))
        out.append((f"pipe_msk_{c['tag']}_k{c['k']}", ndiff(r["mask"][0], c["out_msk"]), 0))
        assert r["image"].is_contiguous(memory_format=torch.channels_last) or r["image"].shape[1] == 1
    # batches with mixed rotations (square), ragged tile edges, per-image /255 decision, against the oracle
    rng = np.random.default_rng(3)
    for tag, (B, H, W, C) in {"sq_gray": (5, 96, 96, 1), "sq_rgb": (4, 70, 70, 3), "rect_odd": (3, 45, 83, 1),
                              "rect_even": (3, 45, 83, 3), "tiny": (2, 1, 1, 1), "one_row": (2, 1, 37, 1)}.items():
        shape = (B, H, W) if C == 1 else (B, H, W, C)
        imgs = rng.integers(0, 256, size=shape, dtype=np.uint8)
        imgs[0] = imgs[0] & 1                                   # image 0 keeps its 0/1 bytes unscaled
        msks = np.array([0, 128, 255, 1, 254], dtype=np.uint8)[rng.integers(0, 5, size=(B, H, W))]
        if tag.startswith("sq"):
            rots = [i % 4 for i in range(B)]
        elif tag == "rect_odd":
            rots = [1, 3, 1]
        elif tag == "rect_even":
            rots = [0, 2, 2]
        else:
            rots = None
        oi, om = IO.make_batch(list(imgs), list(msks), rots or [0] * B)
        r = UD.preprocess_batch(imgs, msks, rots, device=DEV)
        out.append((f"pipe_batch_img_{tag}", ndiff(r["image"], oi), 0))
        out.append((f"pipe_batch_msk_{tag}", ndiff(r["mask"], om), 0))
    # caller-supplied gray-level table
    lut = np.arange(256, dtype=np.int64) // 64
    m = rng.integers(0, 256, size=(2, 33, 65), dtype=np.uint8)
    r = UD.preprocess_batch(np.zeros((2, 33, 65), np.uint8), m, None, device=DEV, lut=lut)
    out.append(("pipe_mask_lut", ndiff(r["mask"], torch.from_numpy(lut[m])), 0))
    return out


def check_pipeline_full_size():
    """BASELINE's batch (16 x 1 x 512 x 512) through a size-independent property: rotating by k on the device equals
    torch.rot90 of the unrotated result, four quarter turns of the mask come back to the start, values = byte / 255."""
    out = []
    g = torch.Generator().manual_seed(9)
    imgs = torch.randint(0, 256, (16, 512, 512), dtype=torch.uint8, generator=g)
    msks = torch.tensor([0, 128, 255], dtype=torch.uint8)[torch.randint(0, 3, (16, 512, 512), generator=g)]
    base = UD.preprocess_batch(imgs, msks, None, device=DEV)
    # true division on the host like numpy's (data_loading.py:87); torch's CUDA `x / 255.0` multiplies by the
    # rounded reciprocal and differs in the last bit for ~half of the byte values
    want = torch.from_numpy(imgs.numpy().astype(np.float32) / 255.0).unsqueeze(1)
    out.append(("pipe_full_values", ndiff(base["image"], want), 0))
    want_m = (msks.to(DEV) == 255).long() * 2 + (msks.to(DEV) == 128).long()
    out.append(("pipe_full_mask", ndiff(base["mask"], want_m), 0))
    for k in (1, 2, 3):
        r = UD.preprocess_batch(imgs, msks, [k] * 16, device=DEV)
        out.append((f"pipe_full_rot{k}_img", ndiff(r["image"], torch.rot90(base["image"], k, dims=(2, 3))), 0))
        out.append((f"pipe_full_rot{k}_msk", ndiff(r["mask"], torch.rot90(base["mask"], k, dims=(1, 2))), 0))
    return out


def _dev_logits(x):
    """the layout the UNet hands over: logical NCHW, physically NHWC"""
    return x.to(DEV).contiguous(memory_format=torch.channels_last)


def check_eval_tail(gio=None):
    gio = gio or load_golden_io()
    out = []
    for c in gio["eval_mc"]:
        for layout in ("nhwc", "nchw"):
            lg = _dev_logits(c["logits"]) if layout == "nhwc" else c["logits"].to(DEV).contiguous()
            for tdt in (torch.float32, torch.int64):
                idx, dice, counts = UE.argmax_class_dice(lg, c["true"].to(DEV).to(tdt), c=c["c"])
                out.append((f"eval_mc_idx_{c['tag']}_{layout}_{tdt}", ndiff(idx, c["idx"]), 0))
                out.append((f"eval_mc_dice_{c['tag']}_{layout}_{tdt}", abs(dice.item() - c["dice"].item()), 1e-6))
                _, _, oc = IO.eval_multiclass(c["logits"], c["true"], c["c"])
                out.append((f"eval_mc_counts_{c['tag']}_{layout}_{tdt}", ndiff(counts[:, :3], oc), 0))
        idx8, _, _ = UE.argmax_class_dice(_dev_logits(c["logits"]), c["true"].to(DEV), c=c["c"], index_dtype=torch.uint8)
        out.append((f"eval_mc_idx_u8_{c['tag']}", ndiff(idx8.long(), c["idx"]), 0))
    for c in gio["eval_bin"]:
        pred, dice, counts = UE.binary_dice(c["logits"].to(DEV), c["true"].to(DEV))
        out.append((f"eval_bin_pred_{c['tag']}", ndiff(pred.float(), c["binary"]), 0))
        out.append((f"eval_bin_dice_{c['tag']}", abs(dice.item() - c["dice"].item()), 1e-6))
        out.append((f"eval_bin_valid_{c['tag']}", float(counts[:, 3].sum().item()), 0))
    # an invalid binary target (evaluate.py:57 asserts) -> NaN dice, counted
    _, dice, counts = UE.binary_dice(torch.zeros(1, 1, 8, 8, device=DEV), torch.full((1, 8, 8), 5.0, device=DEV))
    out.append(("eval_bin_invalid_is_nan", 0.0 if (torch.isnan(dice).item() and counts[0, 3].item() == 64) else 1.0, 0))
    # larger seeded cases against the oracle: bf16 NHWC logits with many exact ties, NaN handling
    g = torch.Generator().manual_seed(21)
    for tag, (B, C, H, W, dt) in {"big_bf16": (4, 3, 256, 320, torch.bfloat16), "big_f32": (2, 4, 200, 120, torch.float32),
                                  "c8": (1, 8, 64, 64, torch.bfloat16)}.items():
        lg = (torch.randn(B, C, H, W, generator=g) * 2).to(dt)
        if tag == "big_f32":
            lg[0, 1, 5, 7] = float("nan")
        true = torch.randint(0, C, (B, H, W), generator=g)
        oi, od, oc = IO.eval_multiclass(lg, true.float(), 2)
        idx, dice, counts = UE.argmax_class_dice(_dev_logits(lg), true.to(DEV), c=2)
        out.append((f"eval_mc_idx_{tag}", ndiff(idx, oi), 0))
        out.append((f"eval_mc_counts_{tag}", ndiff(counts[:, :3], oc), 0))
        out.append((f"eval_mc_dice_{tag}", abs(dice.item() - od.item()), 1e-6))
    return out


def _predict_case(out, tag, logits, size, index_dtype=torch.int64):
    """Three gates per case.  (1) bit-exact against the op-by-op restatement of ATen's CUDA arithmetic (fp32 lambdas,
    value rounded to the storage type, first maximum).  (2) Against the reference expression itself: the CPU fixture /
    CPU ``F.interpolate(...).argmax`` -- exact for fp32 and for the identity resize; for bf16 ATen's *CPU* kernel
    rounds the interpolation weights to bf16 (UpSampleKernel.cpp stores them as scalar_t) while its *CUDA* kernel --
    the one predict.py runs on a GPU -- keeps them in fp32 like ours, so the CPU comparison carries a 5e-3 budget and
    the CUDA comparison (same device, torch's own kernel, FMA contraction the only difference) 2e-4.  (3) Every pixel
    that differs from the argmax of the fp32 interpolation must be a near tie: top-2 margin within the bf16 rounding
    of the two values."""
    import torch.nn.functional as F
    H, W = size
    for layout in ("nhwc", "nchw"):
        lg = _dev_logits(logits) if layout == "nhwc" else logits.to(DEV).contiguous()
        idx = UE.resize_argmax(lg, size, index_dtype=index_dtype).long()
        out.append((f"predict_exact_{tag}_{layout}", ndiff(idx, IO.resize_argmax_exact(logits, size)), 0))
        same = logits.shape[-2:] == (H, W)
        bf = logits.dtype == torch.bfloat16
        dis = 1.0 - (idx.cpu() == IO.predict_tail(logits, size)).float().mean().item()
        out.append((f"predict_ref_cpu_{tag}_{layout}", dis, 0.0 if same else (5e-3 if bf else 1e-4)))
        tidx = F.interpolate(lg, size, mode="bilinear").argmax(dim=1)          # predict.py:26-27 on this device
        dis = 1.0 - (idx == tidx).float().mean().item()
        out.append((f"predict_ref_cuda_{tag}_{layout}", dis, 0.0 if same else 2e-4))
        up32 = F.interpolate(logits.float(), size, mode="bilinear")
        top2 = up32.topk(2, dim=1).values
        wrong = idx.cpu() != up32.argmax(dim=1)
        if wrong.any():
            margin = (top2[:, 0] - top2[:, 1])[wrong]
            budget = (top2[:, 0].abs().maximum(top2[:, 1].abs())[wrong]) * (2.0 ** -7 if bf else 2.0 ** -20) + 1e-7
            out.append((f"predict_near_tie_{tag}_{layout}", (margin / budget).max().item(), 1.0))


def check_predict_tail(gio=None):
    gio = gio or load_golden_io()
    out = []
    for c in gio["predict"]:
        _predict_case(out, c["tag"], c["logits"], c["size"])
        # the committed reference fixture (generated by the reference expression in the build container)
        idx = UE.resize_argmax(_dev_logits(c["logits"]), c["size"])
        dis = 1.0 - (idx.cpu() == c["idx"]).float().mean().item()
        bf = c["logits"].dtype == torch.bfloat16
        out.append((f"predict_fixture_{c['tag']}", dis, 0.0 if c["tag"].startswith("same") else (5e-3 if bf else 1e-4)))
    g = torch.Generator().manual_seed(22)
    for tag, (B, C, h, w, H, W, dt) in {"up_big_bf16": (2, 4, 128, 160, 300, 333, torch.bfloat16),
                                        "same_bf16": (2, 3, 96, 128, 96, 128, torch.bfloat16),
                                        "down_f32": (1, 3, 257, 129, 100, 64, torch.float32)}.items():
        lg = torch.randn(B, C, h, w, generator=g).to(dt)
        _predict_case(out, tag, lg, (H, W), index_dtype=torch.uint8)
    return out


def check_reference_shaped_entry_points():
    """unetb200.eval_tail.evaluate / predict_img on the B200 UNet against the same model's logits pushed through the
    oracle's restatement of the reference tails."""
    import unet
    out = []
    torch.manual_seed(0)
    dev = torch.device(DEV)
    for ncls in (3, 1):
        net = unet.UNet(1, ncls).to(dev).to(memory_format=torch.channels_last)
        g = torch.Generator().manual_seed(31 + ncls)
        batches = [{"image": torch.rand(2, 1, 64, 64, generator=g),
                    "mask": torch.randint(0, 3 if ncls > 1 else 4, (2, 64, 64), generator=g)} for _ in range(3)]
        got = UE.evaluate(net, batches, dev, amp=True)
        net.eval()
        scores = []
        with torch.inference_mode(), torch.autocast("cuda", enabled=True):
            for b in batches:
                lg = net(b["image"].to(dev).contiguous(memory_format=torch.channels_last)).cpu()
                if ncls > 1:
                    scores.append(IO.eval_multiclass(lg, b["mask"].float(), 2)[1].item())
                else:
                    scores.append(IO.eval_binary(lg, b["mask"].float())[1].item())
        net.train()
        out.append((f"evaluate_mean_ncls{ncls}", abs(got[0] - sum(scores) / 3), 1e-6))
        out.append((f"evaluate_post_equals_orig_ncls{ncls}", abs(got[1] - got[0]), 0))
        out.append((f"evaluate_min_ncls{ncls}", abs(got[2] - min(scores)), 1e-6))
        if ncls > 1:
            img = torch.rand(1, 64, 64, generator=g)
            idx = UE.predict_img(net, img, dev, out_size=(80, 100))
            with torch.no_grad(), torch.autocast("cuda", enabled=True):
                lg = net(img.unsqueeze(0).to(dev).contiguous(memory_format=torch.channels_last)).cpu()
            out.append(("predict_img_exact", ndiff(idx, IO.resize_argmax_exact(lg, (80, 100))[0]), 0))
            out.append(("predict_img_mode", 0.0 if not net.training else 1.0, 0))
    return out


GROUPS = {
    "io_pipeline": lambda: check_pipeline(),
    "io_pipeline_full": lambda: check_pipeline_full_size(),
    "eval_tail": lambda: check_eval_tail(),
    "predict_tail": lambda: check_predict_tail(),
    "tail_entry_points": lambda: check_reference_shaped_entry_points(),
}
