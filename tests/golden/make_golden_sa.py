"""Pin the oracle's SpatialAttention / UNet_SA restatement against the UNMODIFIED reference.

    UNETB200_REFERENCE_DIR=<reference checkout> python tests/golden/make_golden_sa.py

Builds the reference's ``UNet_SA`` (unet_model.py:140-189; ``Up(..., use_attention=True)``, unet_parts.py:62-98 with the
``SpatialAttention`` gate of :39-60) under a fixed seed, runs one training step (CE + dice, train.py:137-142) on the
oracle's synthetic batch, asserts the oracle agrees (its ``up`` applies the gate exactly when the state holds the 7x7
weight), and commits ``golden_sa_v1.pt``: per-tensor sums of the seeded state, logits, loss, gradient norms and samples, plus one
stand-alone gate case (x * attention(x) forward / backward) -- re-checked by tests/test_oracle_sa.py without
the reference and used by the -m gpu gate of the CUDA kernels.
"""
import os
import sys

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))


def main():
    from make_golden import _load_ref
    from oracle import unet_oracle as O
    torch.set_num_threads(os.cpu_count())
    refunet, refparts, refdice, _ = _load_ref()
    G = {}
    for tag, (nc, ncls, bil, B, H, W) in {"sa_1_2_convT": (1, 2, False, 2, 64, 64), "sa_3_3_bilinear": (3, 3, True, 1, 48, 80)}.items():
        torch.manual_seed(11)
        ref = sys.modules["refunet.unet_model"].UNet_SA(nc, ncls, bil).train()
        st = {k: v.detach().clone() for k, v in ref.state_dict().items()}
        img, msk = O.synthetic_batch(B, nc, ncls, H, W)
        logits = ref(img)
        loss = F.cross_entropy(logits, msk) + refdice.dice_loss(
            F.softmax(logits, dim=1).float(), F.one_hot(msk, ncls).permute(0, 3, 1, 2).float(), multiclass=True)
        loss.backward()
        grads = {k: p.grad.detach().clone() for k, p in ref.named_parameters()}
        o_logits, o_loss, o_grads = O.training_step({k: v.clone() for k, v in st.items()}, img, msk, ncls, bil)
        e_l = O.rel_err(o_logits, logits)
        e_g = max(O.rel_l2(o_grads[k], grads[k]) for k in grads)
        print(tag, "oracle vs reference UNet_SA: logits max-rel", e_l, "loss", abs(float(o_loss) - float(loss)), "worst grad rel-L2", e_g)
        assert e_l < 1e-5 and abs(float(o_loss) - float(loss)) < 1e-6 and e_g < 2e-4, (tag, e_l, e_g)
        assert set(o_grads) == set(grads)
        # small fixture: the state is re-created from the seed by the drop-in constructor (whose draws must equal the
        # reference's: checked through the per-tensor sums), gradients are pinned by norm + a strided sample
        G[tag] = dict(cfg=(nc, ncls, bil, B, H, W), seed=11, keys=list(st),
                      state_sum={k: v.double().sum() for k, v in st.items()},
                      logits=logits.detach().clone(), loss=loss.detach().clone(),
                      grad_norm={k: g.double().norm() for k, g in grads.items()},
                      grad_sample={k: g.reshape(-1)[:: max(1, g.numel() // 64)][:64].clone() for k, g in grads.items()})
    # stand-alone gate: Up.forward's  x2 = x2 * self.attention(x2)
    torch.manual_seed(12)
    att = refparts.SpatialAttention()
    x = torch.relu(torch.randn(2, 16, 9, 13)).requires_grad_(True)        # post-ReLU like a skip tensor (zeros -> ties)
    y = x * att(x)
    gy = torch.randn_like(y)
    y.backward(gy)
    G["gate"] = dict(w=att.conv1.weight.detach().clone(), x=x.detach().clone(), y=y.detach().clone(), gy=gy,
                     gx=x.grad.clone(), gw=att.conv1.weight.grad.clone())
    out = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden_sa_v1.pt")
    torch.save(G, out)
    print("wrote", out, os.path.getsize(out) / 1e3, "kB")


if __name__ == "__main__":
    main()
