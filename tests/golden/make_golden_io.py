"""Generate tests/golden/golden_io_v1.pt by running the UNMODIFIED reference code either side of the
UNet step (SURVEY.md section 8(f) N1, N3) on seeded synthetic bytes:

    UNETB200_REFERENCE_DIR=<reference checkout> python tests/golden/make_golden_io.py

  * utils/data_loading.py: BasicDataset.preprocess + rotate_image_and_mask (through PIL, as __getitem__ does)
  * utils/dice_score.py:   dice_coeff, applied to the literal tail expressions of evaluate.py:56-66,111-117
  * predict.py:26-27:      F.interpolate(bilinear) + argmax

The script asserts that oracle/io_oracle.py reproduces every fixture it writes.
"""
import importlib.util
import os
import sys

import numpy as np
import torch
import torch.nn.functional as F
from PIL import Image

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
REF = os.environ.get("UNETB200_REFERENCE_DIR") or sys.exit("set UNETB200_REFERENCE_DIR to a checkout of the reference")
sys.path.insert(0, ROOT)


def _load(name, path):
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    sys.modules[name] = mod
    spec.loader.exec_module(mod)
    return mod


def main():
    from oracle import io_oracle as IO
    refdata = _load("refdata", f"{REF}/utils/data_loading.py")
    refdice = _load("refdice_io", f"{REF}/utils/dice_score.py")
    DS = refdata.BasicDataset
    rng = np.random.default_rng(7)
    G = {"pipeline": [], "eval_mc": [], "eval_bin": [], "predict": []}

    # ---- input pipeline: gray and RGB images, masks with legal and stray gray levels, all four rotations
    for tag, (H, W, C, lo_only) in {
        "gray_40x56": (40, 56, 1, False), "rgb_33x47": (33, 47, 3, False), "gray_64x64": (64, 64, 1, False),
        "gray_binary_24x24": (24, 24, 1, True),          # no value > 1: the /255 branch is NOT taken
    }.items():
        img = rng.integers(0, 2 if lo_only else 256, size=(H, W) if C == 1 else (H, W, C), dtype=np.uint8)
        levels = np.array([0, 128, 255, 7, 200], dtype=np.uint8)
        msk = levels[rng.integers(0, 5, size=(H, W))]
        for k in range(4):
            pil_i, pil_m = Image.fromarray(img), Image.fromarray(msk)
            if k:                                               # data_loading.py:119-121
                pil_i, pil_m = DS.rotate_image_and_mask(pil_i, pil_m, [90, 180, 270][k - 1])
            out_i = DS.preprocess(None, pil_i, 1, is_mask=False)
            out_m = DS.preprocess(None, pil_m, 1, is_mask=True)
            ti = torch.as_tensor(out_i.copy()).float().contiguous()      # :130
            tm = torch.as_tensor(out_m.copy()).long().contiguous()       # :131
            oi, om = IO.make_batch([img], [msk], [k])
            assert torch.equal(oi[0], ti) and torch.equal(om[0], tm), (tag, k)
            G["pipeline"].append(dict(tag=tag, k=k, img=torch.from_numpy(img.copy()), msk=torch.from_numpy(msk.copy()),
                                      out_img=ti, out_msk=tm))

    # ---- evaluate tails
    gen = torch.Generator().manual_seed(11)
    for tag, (B, C, H, W, dt) in {"mc_f32": (3, 3, 37, 53, torch.float32), "mc_bf16": (2, 4, 64, 48, torch.bfloat16),
                                  "mc_empty": (2, 3, 16, 16, torch.float32)}.items():
        logits = torch.randn(B, C, H, W, generator=gen).to(dt)
        if dt == torch.bfloat16:
            logits = (logits * 4).round().div(4).to(dt)          # many exact ties between classes
        true = torch.randint(0, 3, (B, H, W), generator=gen).float()
        if tag == "mc_empty":
            logits[:, 2] = -100.0                                # class 2 never predicted ...
            true[true == 2] = 0                                  # ... nor present: sets_sum == 0 branch
        mask_pred = logits
        mask_pred_indices = mask_pred.argmax(dim=1)              # evaluate.py:111
        c = 2
        pred_c = (mask_pred_indices == c).float()
        true_c = (true == c).float()
        dice = refdice.dice_coeff(pred_c, true_c, reduce_batch_first=False)
        oidx, odice, _ = IO.eval_multiclass(logits, true, c)
        assert torch.equal(oidx, mask_pred_indices) and torch.equal(odice, dice), tag
        G["eval_mc"].append(dict(tag=tag, logits=logits, true=true, c=c, idx=mask_pred_indices, dice=dice))
    for tag, (B, H, W, dt) in {"bin_f32": (3, 29, 31, torch.float32), "bin_bf16": (2, 32, 40, torch.bfloat16)}.items():
        logits = (torch.randn(B, 1, H, W, generator=gen) * 0.05).to(dt)     # near the 0.5 threshold
        true = torch.randint(0, 4, (B, H, W), generator=gen).float()
        mask_true = true.clone()
        mask_true //= 2                                                      # evaluate.py:56
        prob = torch.sigmoid(logits.squeeze(1))
        binary = (prob > 0.5).float()
        dice = refdice.dice_coeff(binary, mask_true, reduce_batch_first=False)
        ob, od, _ = IO.eval_binary(logits, true)
        assert torch.equal(ob, binary) and torch.equal(od, dice), tag
        G["eval_bin"].append(dict(tag=tag, logits=logits, true=true, binary=binary, dice=dice))

    # ---- predict tail
    for tag, (B, C, h, w, H, W, dt) in {"same_f32": (1, 3, 40, 56, 40, 56, torch.float32),
                                        "up_f32": (1, 3, 20, 28, 47, 61, torch.float32),
                                        "down_f32": (2, 4, 50, 40, 31, 23, torch.float32),
                                        "up_bf16": (1, 3, 24, 24, 48, 72, torch.bfloat16)}.items():
        logits = torch.randn(B, C, h, w, generator=gen).to(dt)
        up = F.interpolate(logits, (H, W), mode='bilinear')      # predict.py:26
        idx = up.argmax(dim=1)                                   # predict.py:27
        ex = IO.resize_argmax_exact(logits, (H, W))
        agree = (ex == idx).float().mean().item()
        print(f"predict {tag}: restated arithmetic agrees with ATen on {agree:.6f} of pixels")
        assert agree >= (1.0 if tag.startswith("same") else 0.999), tag
        G["predict"].append(dict(tag=tag, logits=logits, size=(H, W), idx=idx))

    for cases in G.values():                    # label maps (values < 256) as uint8: the loaders widen them to int64
        for c in cases:
            for k in ("out_msk", "idx"):
                if k in c:
                    assert 0 <= int(c[k].min()) and int(c[k].max()) < 256, (c["tag"], k)
                    c[k] = c[k].to(torch.uint8)
    out = os.path.join(ROOT, "tests", "golden", "golden_io_v1.pt")
    torch.save(G, out)
    print("wrote", out, os.path.getsize(out), "bytes")


if __name__ == "__main__":
    main()
