"""-m gpu: the binary (n_classes = 1) training path, train.py:118-134.

* the fused BCE-with-logits + sigmoid-dice kernels (``losses.bce_dice_loss``) against a CPU fp64 restatement of
  the autocast composition, over target dtypes, soft / class-index targets, extreme logits and the empty-set case;
  bit-reproducibility;
* full training steps of ``UNet(1, 1)`` / ``UNet_S(1, 1)`` through ``losses.training_criterion``'s binary defaults
  against ``oracle.training_step(..., n_classes=1)``: at random init with the bars of ``gpu_e2e.width_gate``, on a
  well-conditioned state with north_star's bf16 bars;
* whole-step CUDA-graph replays against eager steps.
"""
import os
import statistics

import pytest
import torch
import torch.nn.functional as F

from gpu_checks import BF, DEV, FP, TOL, O, host, rel
from unetb200 import losses as UL

pytestmark = pytest.mark.gpu


# ------------------------------------------------------------------------------------------------
# kernel parity
# ------------------------------------------------------------------------------------------------
class _SigmoidInDtype(torch.autograd.Function):
    """torch.sigmoid of the logits in their storage dtype, on an fp64 graph: the value is rounded like F.sigmoid of
    bf16 logits under autocast, and the gradient is s (1 - s) of that rounded output (sigmoid's autograd formula)."""

    @staticmethod
    def forward(ctx, x64, dtype):
        s = torch.sigmoid(x64.to(dtype)).double()
        ctx.save_for_backward(s)
        return s

    @staticmethod
    def backward(ctx, g):
        (s,) = ctx.saved_tensors
        return g * s * (1 - s), None


def _reference(x, t, gscale=1.0, eps=1e-6):
    """F.binary_cross_entropy_with_logits(x.float(), t) + dice_loss(torch.sigmoid(x).float(), t) in fp64 on the CPU
    (dice_score.py:12-18 on a 3-D input: one global ratio, sets == 0 -> inter).  Returns (total, bce, dice_loss,
    dice) and the gradient of gscale * total with respect to x."""
    x64 = x.detach().double().requires_grad_(True)
    t64 = t.double()
    bce = F.binary_cross_entropy_with_logits(x64, t64)
    s = _SigmoidInDtype.apply(x64, x.dtype)
    inter = 2 * (s * t64).sum()
    sets = s.sum() + t64.sum()
    sets = torch.where(sets == 0, inter, sets)
    dice = (inter + eps) / (sets + eps)
    total = bce + (1 - dice)
    (gscale * total).backward()
    return [float(v.detach()) for v in (total, bce, 1 - dice, dice)], x64.grad


def _logits(shape, dtype, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(shape, generator=g) * 3
    flat = x.view(-1)
    idx = torch.randperm(flat.numel(), generator=g)[:max(4, flat.numel() // 50)]
    flat[idx] = torch.tensor([100.0, -100.0, 60.0, -60.0]).repeat(len(idx) // 4 + 1)[:len(idx)]   # |x| up to 100
    return x.to(dtype)


def _targets(shape, kind, seed):
    g = torch.Generator().manual_seed(seed + 1)
    if kind == "f32":
        return torch.randint(0, 2, shape, generator=g).float()
    if kind == "f32_soft":                         # torch accepts soft targets
        return torch.randint(0, 3, shape, generator=g).float() * 0.3
    hi = 3                                         # class index 2 (a 255 mask pixel before train.py's //= 2)
    if kind == "i64":
        return torch.randint(0, hi, shape, generator=g)
    return torch.randint(0, hi, shape, generator=g).to(torch.uint8)


def _check_parity(x, t, gpu_logits):
    """gpu_logits: the device copy of x in the layout under test (any shape bce_dice_loss accepts)."""
    gs = 1.7
    ref, ref_grad = _reference(x, t, gs)
    lg = gpu_logits.requires_grad_(True)
    total, parts = UL.bce_dice_loss(lg, t.to(DEV), return_parts=True)
    (total * gs).backward()
    got = [float(v) for v in parts.cpu()]
    loss_tol = 2e-6 if x.dtype == FP else 1e-5
    assert abs(float(total) - ref[0]) <= loss_tol * abs(ref[0]), f"loss {float(total)!r} vs {ref[0]!r}"
    assert got[0] == float(total)
    for name, a, b in zip(("bce", "dice_loss", "dice"), got[1:], ref[1:]):
        assert abs(a - b) <= 2e-6, f"{name} {a!r} vs {b!r}"
    assert lg.grad.shape == lg.shape and lg.grad.stride() == lg.stride() and lg.grad.dtype == lg.dtype
    e = rel(host(lg.grad).reshape(ref_grad.shape), ref_grad)
    assert e <= (TOL[BF] if x.dtype == BF else 1e-5), f"gradient max-rel {e:.3e}"


@pytest.mark.parametrize("shape", [(3, 37, 29), (16, 256, 256)], ids=["ragged", "many_blocks"])
@pytest.mark.parametrize("dtype", [FP, BF], ids=["fp32", "bf16"])
@pytest.mark.parametrize("tkind", ["f32", "f32_soft", "i64", "u8"])
def test_bce_dice_parity(shape, dtype, tkind):
    x = _logits(shape, dtype, seed=11)
    t = _targets(shape, tkind, seed=11)
    _check_parity(x, t, x.to(DEV))


@pytest.mark.parametrize("dtype", [FP, BF], ids=["fp32", "bf16"])
def test_bce_dice_layouts(dtype):
    """[B,1,H,W] in NCHW and channels_last (the same pixel order for one channel) keep their strides in the
    gradient; a non-contiguous [B,H,W] view is made contiguous first."""
    B, H, W = 2, 45, 52
    x = _logits((B, 1, H, W), dtype, seed=3)
    t = _targets((B, H, W), "f32", seed=3)
    _check_parity(x.squeeze(1), t, x.to(DEV))
    _check_parity(x.squeeze(1), t, x.to(DEV).contiguous(memory_format=torch.channels_last))
    _check_parity(x.squeeze(1), t, x.squeeze(1).transpose(1, 2).contiguous().to(DEV).transpose(1, 2))


@pytest.mark.parametrize("dtype", [FP, BF], ids=["fp32", "bf16"])
def test_bce_dice_empty_sets(dtype):
    """All logits <= -89 (sigmoid underflows to 0) and all targets 0: sets == 0 -> inter, so dice = 1 and the dice
    term contributes no gradient.  The loss itself is ~1e-39, so it is compared in absolute terms."""
    g = torch.Generator().manual_seed(4)
    x = (-89.0 - 10 * torch.rand(2, 33, 40, generator=g)).to(dtype)
    t = torch.zeros(2, 33, 40)
    assert float(torch.sigmoid(x).float().sum()) == 0.0
    ref, ref_grad = _reference(x, t, 1.7)
    lg = x.to(DEV).requires_grad_(True)
    total, parts = UL.bce_dice_loss(lg, t.to(DEV), return_parts=True)
    (total * 1.7).backward()
    got = [float(v) for v in parts.cpu()]
    assert got[3] == 1.0 and got[2] == 0.0
    assert all(abs(a - b) <= 2e-6 for a, b in zip(got, ref))
    gr = host(lg.grad)
    assert bool(torch.isfinite(gr).all()) and float((gr.double() - ref_grad).abs().max()) <= 1e-12


def test_reference_matches_oracle():
    """The composition above is oracle.train_loss(..., n_classes=1) without its boundary term."""
    g = torch.Generator().manual_seed(8)
    lg = torch.randn(2, 1, 24, 40, generator=g) * 2
    t = torch.randint(0, 2, (2, 24, 40), generator=g)
    ref, _ = _reference(lg.squeeze(1), t.float())
    oracle = O.train_loss(lg, t, 1) - 0.25 * O.boundary_loss(lg.squeeze(1), t.float(), edge_width=51, edge_weight=15)
    assert abs(float(oracle) - ref[0]) <= 2e-6 * abs(ref[0])


def test_bce_dice_reproducible():
    x = _logits((16, 256, 256), BF, seed=5).to(DEV)
    t = _targets((16, 256, 256), "f32", seed=5).to(DEV)
    runs = []
    for _ in range(2):
        lg = x.clone().requires_grad_(True)
        total, parts = UL.bce_dice_loss(lg, t, return_parts=True)
        total.backward()
        runs.append((parts.clone(), lg.grad))
    assert torch.equal(runs[0][0], runs[1][0]) and torch.equal(runs[0][1], runs[1][1])


def test_bce_dice_rejects_bad_shapes():
    x = torch.zeros(2, 1, 8, 8, device=DEV)
    with pytest.raises(ValueError):
        UL.bce_dice_loss(x, torch.zeros(2, 8, 9, device=DEV))
    with pytest.raises(ValueError):
        UL.bce_dice_loss(torch.zeros(2, 2, 8, 8, device=DEV), torch.zeros(2, 8, 8, device=DEV))


def test_training_criterion_branches():
    """One channel: bce_dice + 0.25 * boundary(51, 15); more: ce_dice + 0.2 * boundary(51, 7); explicit values win."""
    g = torch.Generator().manual_seed(6)
    t = torch.randint(0, 2, (2, 64, 64), generator=g).to(DEV)
    lg1 = (torch.randn(2, 1, 64, 64, generator=g) * 20).to(DEV)
    lg2 = (torch.randn(2, 2, 64, 64, generator=g) * 20).to(DEV)

    def close(a, b):            # ce_dice sums with fp64 atomics: equal up to the last bit, not bit for bit
        return abs(float(a) - float(b)) <= 1e-6 * abs(float(b))
    bd = UL.bce_dice_loss(lg1, t)
    assert close(UL.training_criterion(lg1, t), bd + 0.25 * UL.boundary_loss(lg1, t, edge_width=51, edge_weight=15))
    assert close(UL.training_criterion(lg1, t, boundary_coeff=0), bd)
    assert close(UL.training_criterion(lg1, t, 0.5, 20, 3), bd + 0.5 * UL.boundary_loss(lg1, t, 20, 3))
    assert close(UL.training_criterion(lg2, t), UL.ce_dice_loss(lg2, t) + 0.2 * UL.boundary_loss(lg2, t, 51, 7))


# ------------------------------------------------------------------------------------------------
# full training steps against the oracle
# ------------------------------------------------------------------------------------------------
# gpu_e2e.width_gate's bars, argmax mismatch read as logit-sign mismatch for one channel
STEP_LIM = {"fp32": dict(logits_maxrel=1e-3, loss_rel=1e-5, sign_mismatch=1e-3, grad_l2_median=2e-2, grad_l2_worst=1e-1),
            "tf32": dict(logits_maxrel=2e-2, loss_rel=1e-3, sign_mismatch=1e-2, grad_l2_median=2e-1, grad_l2_worst=6e-1),
            "bf16": dict(logits_maxrel=1e-1, loss_rel=5e-3, sign_mismatch=3e-2, grad_l2_median=6e-1, grad_l2_worst=1.5)}


def _binary_step(model, img, msk, mode):
    """One training step through training_criterion's binary defaults (0.25 * boundary(51, 15), like
    oracle.train_loss with n_classes=1)."""
    model.zero_grad(set_to_none=True)
    os.environ["UNET_B200_PRECISION"] = "tf32" if mode == "tf32" else "fp32"
    try:
        x = img.to(DEV).contiguous(memory_format=torch.channels_last)
        with torch.autocast("cuda", enabled=(mode == "bf16")):
            logits = model(x)
            loss = UL.training_criterion(logits, msk.to(DEV))
        loss.backward()
    finally:
        os.environ["UNET_B200_PRECISION"] = "fp32"
    return host(logits), float(loss), {k: host(p.grad) for k, p in model.named_parameters()}


def _model(cls_name, st):
    import unet.unet_model as UM
    m = getattr(UM, cls_name)(1, 1)
    m.load_state_dict(st)
    return m.to(DEV).to(memory_format=torch.channels_last).train()


@pytest.mark.parametrize("cls_name,B,H,W,mode", [
    ("UNet", 2, 64, 64, "fp32"), ("UNet", 2, 128, 128, "tf32"), ("UNet", 2, 128, 128, "bf16"),
    ("UNet_S", 2, 128, 128, "bf16"), ("UNet", 2, 100, 84, "fp32")])
def test_binary_step_against_oracle(cls_name, B, H, W, mode):
    import unet.unet_model as UM
    torch.manual_seed(7)
    st = {k: v.detach().clone() for k, v in getattr(UM, cls_name)(1, 1).state_dict().items()}
    img, msk = O.synthetic_batch(B, 1, 1, H, W)
    ref_st = {k: v.clone() for k, v in st.items()}
    r_logits, r_loss, r_grads = O.training_step(ref_st, img, msk, 1)
    model = _model(cls_name, st)
    logits, loss, grads = _binary_step(model, img, msk, mode)
    l2 = [O.rel_l2(grads[k], r_grads[k]) for k in r_grads]
    err = {"logits_maxrel": rel(logits, r_logits),
           "loss_rel": abs(loss - float(r_loss)) / abs(float(r_loss)),
           "sign_mismatch": ((logits > 0) != (r_logits > 0)).float().mean().item(),
           "grad_l2_median": statistics.median(l2), "grad_l2_worst": max(l2)}
    sd = model.state_dict()
    err["running_stats"] = max(rel(host(sd[k]), ref_st[k]) for k in sd if "running" in k)
    lim = dict(STEP_LIM[mode], running_stats=1e-4 if mode == "fp32" else 2e-2)
    bad = {k: (v, lim[k]) for k, v in err.items() if not v <= lim[k]}
    assert not bad, f"{cls_name} {B}x{H}x{W} {mode}: {bad}"


_COND = {}


def _conditioned_binary_state():
    """Like oracle.conditioned_state, for one output channel: ten fp32 CPU steps of the reference's binary
    arithmetic (oracle.training_step with n_classes=1, plain RMSprop alpha 0.99 eps 1e-8, lr 1e-3) on {0,1}
    contour masks.  structured_batch(..., n_classes=1) draws no foreground, so the masks come from n_classes=2."""
    if "st" not in _COND:
        st = O.build_state(1, 1, False, seed=0)
        img, msk = O.structured_batch(2, 1, 2, 128, 128)
        names = O.param_names(st)
        sq = {k: torch.zeros_like(st[k]) for k in names}
        for _ in range(10):
            _, _, g = O.training_step(st, img, msk, 1)
            for k in names:
                sq[k].mul_(0.99).addcmul_(g[k], g[k], value=1 - 0.99)
                st[k] = st[k].addcdiv(g[k], sq[k].sqrt().add_(1e-8), value=-1e-3)
        _COND["st"] = st
    return {k: v.clone() for k, v in _COND["st"].items()}


def test_binary_bf16_conditioned_north_star():
    """north_star's bf16 bars on a well-conditioned binary state: logits and gradients within 2e-2, loss and dice
    within 1e-3, >= 99.9 % of the pixels thresholded alike."""
    st = _conditioned_binary_state()
    img, msk = O.structured_batch(2, 1, 2, 128, 128, seed=9)
    names = O.param_names(st)
    r_logits, r_loss, r_grads = O.training_step({k: v.clone() for k, v in st.items()}, img, msk, 1)
    logits, loss, grads = _binary_step(_model("UNet", st), img, msk, "bf16")
    dice = lambda lg: float(O.dice_coeff(torch.sigmoid(lg.squeeze(1)), msk.float(), True))  # noqa: E731
    cat = lambda g: torch.cat([g[k].reshape(-1).double() for k in names])  # noqa: E731
    l2 = [O.rel_l2(grads[k], r_grads[k]) for k in names]
    err = {"logits_maxrel": (rel(logits, r_logits), 2e-2),
           "loss_rel": (abs(loss - float(r_loss)) / abs(float(r_loss)), 1e-3),
           "dice_abs": (abs(dice(logits) - dice(r_logits)), 1e-3),
           "sign_mismatch": (((logits > 0) != (r_logits > 0)).float().mean().item(), 1e-3),
           "grad_all_rel_l2": (O.rel_l2(cat(grads), cat(r_grads)), 2e-2),
           "grad_l2_median": (statistics.median(l2), 2e-2),
           "grad_maxrel_median": (statistics.median(rel(grads[k], r_grads[k]) for k in names), 2e-2),
           # north_star_gate's per-tensor worst case below 4 x 256 x 256 pixels
           "grad_l2_worst": (max(l2), 1e-1)}
    bad = {k: v for k, v in err.items() if not v[0] <= v[1]}
    assert not bad, f"binary conditioned bf16: {bad}"


# ------------------------------------------------------------------------------------------------
# CUDA graphs
# ------------------------------------------------------------------------------------------------
def test_binary_graph_replays_match_eager():
    """GraphedStep with FusedRMSprop(clip_max_norm=1.0) on UNet(1, 1), bf16: after the same two warm-up steps,
    three replays and three eager steps give the same losses and parameters (the bars of gpu_e2e.graph_gate)."""
    from unetb200.graph import GraphedStep
    from unetb200.optim import FusedRMSprop
    torch.manual_seed(7)
    import unet
    st = {k: v.detach().clone() for k, v in unet.UNet(1, 1).state_dict().items()}
    img, msk = O.synthetic_batch(2, 1, 1, 64, 64)
    x = img.to(DEV).contiguous(memory_format=torch.channels_last)
    t = msk.to(DEV)

    def make():
        m = _model("UNet", st)
        opt = FusedRMSprop(m.parameters(), lr=1e-4)

        def step(xx, tt):
            for p in m.parameters():
                p.grad = None
            with torch.autocast("cuda", enabled=True):
                loss = UL.training_criterion(m(xx), tt)
            loss.backward()
            opt.step(clip_max_norm=1.0)
            return loss
        return m, step

    m1, step1 = make()
    eager = [float(step1(x, t).detach()) for _ in range(5)]
    m2, step2 = make()
    g = GraphedStep(step2, (x, t), warmup=2)
    replayed = [float(g.replay()) for _ in range(3)]
    torch.cuda.synchronize()
    assert all(v == v and abs(v) < 1e3 for v in eager + replayed), (eager, replayed)
    # gpu_e2e.graph_gate's bars: a bf16 ReLU-mask flip may move later steps, a race gives NaN or errors >> 1
    for a, b, tol in zip(replayed, eager[2:], (2e-3, 5e-3, 5e-3)):
        assert abs(a - b) <= tol * abs(b), (replayed, eager)
    w1 = {k: host(v) for k, v in m1.state_dict().items() if v.dtype.is_floating_point}
    w2 = {k: host(v) for k, v in m2.state_dict().items() if v.dtype.is_floating_point}
    assert max(O.rel_l2(w2[k], w1[k]) for k in w1 if "running" not in k and not k.endswith(".bias")) <= 1e-2
    assert max(float((w2[k] - w1[k]).abs().max()) for k in w1 if k.endswith(".bias")) <= 1e-3
