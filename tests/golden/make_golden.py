"""Generate tests/golden/*.pt by running the UNMODIFIED reference (imported read-only from the checkout that
UNETB200_REFERENCE_DIR names) on seeded synthetic inputs:

    UNETB200_REFERENCE_DIR=<reference checkout> python tests/golden/make_golden.py

The tests read the committed fixtures and never need the reference.  The script also
asserts, bit for bit, that oracle.build_state() draws the same weights as the reference
constructor, and that the oracle reproduces every fixture it writes (so a fixture can never be
committed that the oracle disagrees with).
"""
import os
import sys
import types

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
REF = os.environ.get("UNETB200_REFERENCE_DIR") or sys.exit("set UNETB200_REFERENCE_DIR to a checkout of the reference")
sys.path.insert(0, ROOT)

# import the reference's own modules under private names so they cannot shadow anything
def _load_ref():
    import importlib.util

    def load(name, path, pkg_path=None):
        spec = importlib.util.spec_from_file_location(name, path, submodule_search_locations=pkg_path)
        mod = importlib.util.module_from_spec(spec)
        sys.modules[name] = mod
        spec.loader.exec_module(mod)
        return mod
    unet = load("refunet", f"{REF}/unet/__init__.py", [f"{REF}/unet"])
    dice = load("refdice", f"{REF}/utils/dice_score.py")
    bnd = load("refboundary", f"{REF}/utils/boundary_loss.py")
    return unet, sys.modules["refunet.unet_parts"], dice, bnd


def main():
    from oracle import unet_oracle as O
    torch.set_num_threads(os.cpu_count())
    refunet, refparts, refdice, refbnd = _load_ref()
    G = {}

    # ---- 1. constructor parity + full-network step fixtures ---------------------------------
    for tag, (nc, ncls, bil, B, H, W) in {
        "unet_1_2_convT_32": (1, 2, False, 2, 32, 32),
        "unet_1_2_bilinear_32": (1, 2, True, 2, 32, 32),
        "unet_3_4_convT_48": (3, 4, False, 1, 48, 48),
        "unet_1_2_convT_256_C1": (1, 2, False, 1, 256, 256),      # BASELINE.json configs[0]
    }.items():
        torch.manual_seed(0)
        ref = refunet.UNet(nc, ncls, bil)
        st = O.build_state(nc, ncls, bil, seed=0)
        rsd = ref.state_dict()
        assert list(rsd.keys()) == list(st.keys()), "state_dict key order differs"
        for k in rsd:
            assert torch.equal(rsd[k], st[k]), f"constructor draw differs at {k}"
        img, msk = O.synthetic_batch(B, nc, ncls, H, W)
        ref.train()
        logits = ref(img)
        # train.py:137-142
        loss = F.cross_entropy(logits, msk)
        loss = loss + refdice.dice_loss(F.softmax(logits, dim=1).float(),
                                        F.one_hot(msk, ncls).permute(0, 3, 1, 2).float(), multiclass=True)
        bl = refbnd.boundary_loss(logits, msk.float(), edge_width=5, edge_weight=7)
        (loss + 0.2 * bl).backward()
        assert not bl.requires_grad
        o_logits, o_loss, o_grads = O.training_step(st, img, msk, ncls, bil, boundary_coeff=0.0)
        assert O.rel_err(o_logits, logits) < 1e-5, (tag, O.rel_err(o_logits, logits))
        assert abs(o_loss.item() - loss.item()) < 1e-6
        entry = {"loss": loss.detach(), "boundary": bl.detach(),
                 "logits": logits.detach().clone() if H <= 48 else logits.detach()[:, :, ::8, ::8].clone(),
                 "logits_absmax": logits.detach().abs().max(), "grad_norm": {}, "grad_head": {},
                 "running": {}, "param_sum": {}}
        for k, p in ref.named_parameters():
            g = p.grad
            assert O.rel_err(o_grads[k], g) < 2e-4, (tag, k, O.rel_err(o_grads[k], g))
            entry["grad_norm"][k] = g.norm().double()
            entry["grad_head"][k] = g.reshape(-1)[:32].clone()
            entry["param_sum"][k] = p.detach().double().sum()
        for k, v in ref.state_dict().items():
            if "running" in k or "tracked" in k:
                assert torch.allclose(v.float(), st[k].float(), rtol=1e-5, atol=1e-6), k
                if v.numel() <= 64:
                    entry["running"][k] = v.clone()
        for k in ("outc.conv.weight", "outc.conv.bias", "inc.double_conv.0.weight",
                  "inc.double_conv.1.weight", "inc.double_conv.1.bias"):
            entry["grad_full_" + k] = dict(ref.named_parameters())[k].grad.clone()
        G[tag] = entry
        print(tag, "loss", loss.item(), "boundary", bl.item())

    # ---- 2. per-part fixtures (small channel counts; full tensors) ---------------------------
    def part_fixture(tag, mod, inputs):
        torch.manual_seed(7)
        for p in mod.parameters():
            with torch.no_grad():
                p.copy_(torch.randn_like(p) * 0.3)
        ins = [t.clone().requires_grad_(True) for t in inputs]
        mod.train()
        out = mod(*ins)
        gout = torch.randn(out.shape, generator=torch.Generator().manual_seed(11))
        out.backward(gout)
        G[tag] = {"inputs": [t.detach() for t in inputs], "out": out.detach(), "gout": gout,
                  "gin": [t.grad.clone() for t in ins],
                  "state": {k: v.clone() for k, v in mod.state_dict().items()},
                  "gparams": {k: p.grad.clone() for k, p in mod.named_parameters()}}
        print(tag, tuple(out.shape))

    g = torch.Generator().manual_seed(3)
    part_fixture("DoubleConv_4_8", refparts.DoubleConv(4, 8), [torch.randn(2, 4, 10, 12, generator=g)])
    part_fixture("DoubleConv_4_8_mid6", refparts.DoubleConv(4, 8, 6), [torch.randn(2, 4, 9, 7, generator=g)])
    part_fixture("Down_4_8", refparts.Down(4, 8), [torch.randn(2, 4, 12, 16, generator=g)])
    part_fixture("Down_4_8_odd", refparts.Down(4, 8), [torch.randn(1, 4, 11, 13, generator=g)])
    part_fixture("Up_8_4_convT", refparts.Up(8, 4, bilinear=False),
                 [torch.randn(2, 8, 6, 5, generator=g), torch.randn(2, 4, 12, 10, generator=g)])
    part_fixture("Up_8_4_convT_pad", refparts.Up(8, 4, bilinear=False),
                 [torch.randn(2, 8, 6, 5, generator=g), torch.randn(2, 4, 13, 11, generator=g)])
    part_fixture("Up_8_4_bilinear", refparts.Up(8, 4, bilinear=True),
                 [torch.randn(2, 4, 6, 5, generator=g), torch.randn(2, 4, 12, 10, generator=g)])
    part_fixture("Up_8_4_bilinear_pad", refparts.Up(8, 4, bilinear=True),
                 [torch.randn(2, 4, 6, 5, generator=g), torch.randn(2, 4, 13, 12, generator=g)])
    part_fixture("OutConv_8_3", refparts.OutConv(8, 3), [torch.randn(2, 8, 7, 9, generator=g)])

    # ---- 3. dice ------------------------------------------------------------------------------
    g = torch.Generator().manual_seed(5)
    cases = []
    p4 = torch.softmax(torch.randn(3, 4, 9, 11, generator=g), dim=1)
    t4 = F.one_hot(torch.randint(0, 4, (3, 9, 11), generator=g), 4).permute(0, 3, 1, 2).float()
    cases.append(("mc_loss", p4, t4, dict(multiclass=True)))
    p3 = torch.rand(3, 9, 11, generator=g)
    t3 = (torch.rand(3, 9, 11, generator=g) > 0.5).float()
    cases.append(("bin_loss", p3, t3, dict(multiclass=False)))
    cases.append(("zero_loss", torch.zeros(2, 5, 5), torch.zeros(2, 5, 5), dict(multiclass=False)))
    G["dice"] = {}
    for name, a, b, kw in cases:
        a_ = a.clone().requires_grad_(True)
        v = refdice.dice_loss(a_, b, **kw)
        v.backward()
        G["dice"][name] = {"input": a, "target": b, "multiclass": kw["multiclass"], "loss": v.detach(),
                           "grad": a_.grad.clone()}
        assert abs(O.dice_loss(a, b, **kw).item() - v.item()) < 1e-7
    c = refdice.dice_coeff(p3, t3, reduce_batch_first=False)
    G["dice"]["coeff_nobatch"] = {"input": p3, "target": t3, "value": c}
    c2 = refdice.dice_coeff((p3 > 2).float(), t3 * 0, reduce_batch_first=False)      # empty sets -> 1.0
    G["dice"]["coeff_empty"] = {"input": (p3 > 2).float(), "target": t3 * 0, "value": c2}
    mc = refdice.multiclass_dice_coeff(p4, t4, reduce_batch_first=False)
    G["dice"]["mc_coeff_nobatch"] = {"input": p4, "target": t4, "value": mc}

    # ---- 4. boundary loss -----------------------------------------------------------------------
    G["boundary"] = {}
    g = torch.Generator().manual_seed(9)
    H = W = 40
    yy, xx = torch.meshgrid(torch.arange(H), torch.arange(W), indexing="ij")
    disk = (((yy - 18) ** 2 + (xx - 22) ** 2) < 100)
    tgt255 = torch.zeros(3, H, W)
    tgt255[0][disk] = 255
    tgt255[1][((yy - 5) ** 2 + (xx - 4) ** 2) < 30] = 255
    tgt255[1][((yy - 30) ** 2 + (xx - 30) ** 2) < 50] = 128
    tgt255[2][:, 20:] = 255
    tgt_idx = torch.randint(0, 2, (3, H, W), generator=g).float()
    logits4 = torch.randn(3, 2, H, W, generator=g) * 8            # |x| > 10 occurs -> sigmoid branch
    logits_small = torch.randn(3, 2, H, W, generator=g) * 0.9     # stays inside [-10, 10] -> raw > 0.5
    prob3 = torch.rand(3, H, W, generator=g)
    for name, pred, tgt, ew, wt in (
        ("logits_255", logits4, tgt255, 6, 7.0), ("logits_idx", logits4, tgt_idx, 6, 7.0),
        ("small_255", logits_small, tgt255, 9, 5.0), ("prob3_255", prob3, tgt255, 4, 15.0),
        ("prob3_ew0", prob3, tgt255, 0, 5.0), ("prob3_ew_big", prob3, tgt255, 20, 5.0),
        ("prob3_ew_huge", prob3, tgt255, 64, 5.0), ("single_ch", logits4[:, :1], tgt255, 3, 2.0),
    ):
        v = refbnd.boundary_loss(pred, tgt, edge_width=ew, edge_weight=wt)
        assert not v.requires_grad
        lit = O.boundary_loss(pred, tgt, ew, wt)
        cf = O.boundary_loss_counts(pred, tgt, ew, wt)
        assert abs(lit.item() - v.item()) < 1e-6 and abs(cf - v.item()) < 2e-6, (name, v.item(), lit.item(), cf)
        G["boundary"][name] = {"pred": pred, "target": tgt, "edge_width": ew, "edge_weight": wt,
                               "value": v.clone(), "counts": O.boundary_counts(pred, tgt, ew)}
        print("boundary", name, v.item(), G["boundary"][name]["counts"])
    G["boundary"]["bce_constants"] = torch.tensor(O._bce_constants(), dtype=torch.float64)

    out = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden_v1.pt")
    torch.save(G, out)
    print("wrote", out, os.path.getsize(out) / 1e6, "MB")


if __name__ == "__main__":
    main()
