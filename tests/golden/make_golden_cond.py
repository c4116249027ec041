"""Pin oracle.conditioned_state / structured_batch / Rounding against the UNMODIFIED reference.

    UNETB200_REFERENCE_DIR=<reference checkout> python tests/golden/make_golden_cond.py

The reference's own ``UNet`` module is trained for the same number of steps with ``torch.optim.RMSprop`` on the same
structured batch; the script asserts the oracle's recipe lands on the same state BIT FOR BIT (the recipe restates the
optimizer's single-tensor update op for op: the trajectory is chaotic, a one-ulp difference grows to 1e-1 in ten
steps), then commits a small fingerprint (``golden_cond_v1.pt``: per-tensor sums of the conditioned state, logits
samples, loss, accuracy and gradient norms of one further step on a fresh batch) that ``tests/test_oracle_cond.py``
re-checks on every run without the reference.
"""
import os
import sys

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

CASES = {"cond_1_2_convT": (1, 2, False), "cond_1_2_bilinear": (1, 2, True), "cond_3_4_convT": (3, 4, False)}
STEPS, LR, SIZE, BATCH = 10, 1e-3, 128, 2


def main():
    from make_golden import _load_ref
    from oracle import unet_oracle as O
    torch.set_num_threads(os.cpu_count())
    refunet, _, refdice, _ = _load_ref()
    G = {"recipe": dict(steps=STEPS, lr=LR, size=SIZE, batch=BATCH)}
    for tag, (nc, ncls, bil) in CASES.items():
        torch.manual_seed(0)
        ref = refunet.UNet(nc, ncls, bil).train()
        img, msk = O.structured_batch(BATCH, nc, ncls, SIZE, SIZE)
        opt = torch.optim.RMSprop(ref.parameters(), lr=LR, alpha=0.99, eps=1e-8, foreach=False)
        for _ in range(STEPS):
            opt.zero_grad(set_to_none=True)
            logits = ref(img)
            loss = F.cross_entropy(logits, msk) + refdice.dice_loss(
                F.softmax(logits, dim=1).float(), F.one_hot(msk, ncls).permute(0, 3, 1, 2).float(), multiclass=True)
            loss.backward()
            opt.step()
        st = O.conditioned_state(nc, ncls, bil, STEPS, LR, SIZE, BATCH)
        rsd = {k: v.detach().clone() for k, v in ref.state_dict().items()}   # (the live dict moves with the next forward)
        worst = 0.0
        for k in rsd:
            if rsd[k].dtype.is_floating_point:
                worst = max(worst, O.rel_err(st[k], rsd[k]))
            else:
                assert int(rsd[k]) == int(st[k]), k
        print(tag, "oracle recipe vs reference + torch RMSprop: worst state max-rel", worst)
        assert worst < 2e-4, (tag, worst)
        # one more step from the conditioned state on a fresh structured batch: the fixture the tests compare with
        img2, msk2 = O.structured_batch(BATCH, nc, ncls, SIZE, SIZE, seed=9)
        ref.zero_grad(set_to_none=True)
        logits = ref(img2)
        loss = F.cross_entropy(logits, msk2) + refdice.dice_loss(
            F.softmax(logits, dim=1).float(), F.one_hot(msk2, ncls).permute(0, 3, 1, 2).float(), multiclass=True)
        loss.backward()
        o_logits, o_loss, o_grads = O.training_step({k: v.clone() for k, v in st.items()}, img2, msk2, ncls, bil)
        assert O.rel_err(o_logits, logits) < 5e-4, O.rel_err(o_logits, logits)
        acc = (logits.argmax(1) == msk2).float().mean().item()
        print(tag, "fresh-batch loss", loss.item(), "pixel accuracy", acc)
        G[tag] = {
            "state_sum": {k: v.double().sum() for k, v in rsd.items()},
            "state_absmax": {k: v.double().abs().max() for k, v in rsd.items()},
            "bn_bias_absmax": max(v.abs().max().item() for k, v in rsd.items() if k.endswith(".bias") and v.dim() == 1),
            "loss": loss.detach(), "accuracy": acc, "logits_sample": logits.detach()[:, :, ::8, ::8].clone(),
            "grad_norm": {k: p.grad.norm().double() for k, p in ref.named_parameters()},
        }
    out = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden_cond_v1.pt")
    torch.save(G, out)
    print("wrote", out, os.path.getsize(out) / 1e3, "kB")


if __name__ == "__main__":
    main()
