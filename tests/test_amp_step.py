"""torch.amp.GradScaler and learning-rate schedules with FusedRMSprop, eagerly and inside captured steps.

The reference's step (train.py:80-85,154-159) is RMSprop + CosineAnnealingWarmRestarts + GradScaler in the order
scale(loss).backward(), unscale_, clip_grad_norm_, step, update.  FusedRMSprop takes a 0-dim CUDA tensor ``lr`` (read
by the kernel, so a replayed graph follows the scheduler) and handles GradScaler's ``grad_scale`` / ``found_inf`` on
the device (no host sync, a skipped step stores nothing).

* CPU: validation of ``lr`` and the other hyper-parameters; the optimizer advertises ``_step_supports_amp_scaling``.
* GPU, optimizer level: 12 steps over synthetic gradients with the shapes of UNet(1, 2)'s 64 parameters against
  ``torch.optim.RMSprop(foreach=True)`` + GradScaler, in train.py's order and in the folded form
  ``scaler.step(opt, clip_max_norm=...)``, with a float lr and with tensor lrs driven by two schedulers; inf and NaN
  gradients on two steps.  A direct ``opt.step()`` with only ``grad_scale`` set.  No host sync in the folded step.
* GPU, end to end: bf16 GraphedStep / SegmentedStep replays with GradScaler and a scheduled tensor lr against eager
  steps of the same code, one batch carrying a NaN pixel.
"""
import math
import socket

import pytest
import torch
import torch.distributed as dist

DEV = "cuda"
OPT_TOL = 1e-5         # the rmsprop_* checks of tests/gpu_checks.py
GRAPH_TOL = 1e-6       # graph replay against eager, tests/test_graph_state.py
INJECT = {4: float("inf"), 9: float("nan")}


def _maxrel(a, b):
    from oracle import unet_oracle as O
    return O.rel_err(a, b)


# ------------------------------------------------------------------------------------------------
# CPU
# ------------------------------------------------------------------------------------------------
def _cpu_params():
    return [torch.nn.Parameter(torch.zeros(4, 3)), torch.nn.Parameter(torch.zeros(5))]


@pytest.mark.parametrize("lr,match", [
    (torch.tensor([1e-3], dtype=torch.float32), "0-dim"),
    (torch.tensor(1e-3, dtype=torch.float64), "float32"),
    (torch.tensor(1e-3, dtype=torch.float32), "CUDA"),
])
def test_tensor_lr_validation(lr, match):
    from unetb200.optim import FusedRMSprop
    with pytest.raises(ValueError, match=match):
        FusedRMSprop(_cpu_params(), lr=lr)


@pytest.mark.parametrize("name", ["alpha", "eps", "weight_decay", "momentum"])
def test_tensor_hyper_parameters_rejected(name):
    from unetb200.optim import FusedRMSprop
    with pytest.raises(ValueError, match=name):
        FusedRMSprop(_cpu_params(), lr=1e-3, **{name: torch.tensor(0.5)})


def test_a_group_added_later_is_validated_at_step():
    from unetb200.optim import FusedRMSprop
    opt = FusedRMSprop(_cpu_params(), lr=1e-3)
    opt.add_param_group({"params": [torch.nn.Parameter(torch.zeros(2))], "momentum": torch.tensor(0.9)})
    with pytest.raises(ValueError, match="momentum"):
        opt.step()


def test_supports_amp_scaling():
    from unetb200.optim import FusedRMSprop
    assert FusedRMSprop._step_supports_amp_scaling is True
    assert FusedRMSprop(_cpu_params(), lr=1e-3)._step_supports_amp_scaling


# ------------------------------------------------------------------------------------------------
# GPU, optimizer level
# ------------------------------------------------------------------------------------------------
def _unet_weights(seed=0):
    import unet
    g = torch.Generator().manual_seed(seed)
    return [torch.randn(p.shape, generator=g) * 0.05 for p in unet.UNet(1, 2).parameters()]


def _schedulers(opt, kind):
    S = torch.optim.lr_scheduler
    if kind == "cosine":
        return S.CosineAnnealingWarmRestarts(opt, T_0=4, eta_min=1e-5)
    if kind == "plateau":
        return S.ReduceLROnPlateau(opt, mode="min", factor=0.5, patience=0)
    return None


def _sched_step(s, it):
    if isinstance(s, torch.optim.lr_scheduler.ReduceLROnPlateau):
        s.step(10.0 - it // 2)                 # improves every other step: the LR halves on the others
    elif s is not None:
        s.step()


def _state(opt, ps):
    out = [p.detach().clone() for p in ps]
    for p in ps:
        st = opt.state[p]
        out += [st["square_avg"].clone(), st["momentum_buffer"].clone(), st["step"].clone()]
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("lr_kind", ["float", "cosine", "plateau"])
@pytest.mark.parametrize("order", ["train_py", "folded"])
def test_grad_scaler_matches_torch(order, lr_kind):
    """FusedRMSprop + GradScaler against torch.optim.RMSprop(foreach=True) + GradScaler in train.py's order, over 12
    steps with growth_interval=3, weight decay and momentum 0.999; inf at step 4 and NaN at step 9 in one gradient
    element leave parameters and state bit-identical, halve the scale, and it grows again after 3 clean steps."""
    from unetb200.optim import FusedRMSprop
    ws = _unet_weights()
    pa = [torch.nn.Parameter(w.to(DEV)) for w in ws]
    pb = [torch.nn.Parameter(w.to(DEV)) for w in ws]
    hyper = dict(alpha=0.99, eps=1e-8, weight_decay=1e-4, momentum=0.999)
    oa = torch.optim.RMSprop(pa, lr=1e-3, foreach=True, **hyper)
    lr_b = 1e-3 if lr_kind == "float" else torch.tensor(1e-3, dtype=torch.float32, device=DEV)
    ob = FusedRMSprop(pb, lr=lr_b, **hyper)
    sa = torch.amp.GradScaler("cuda", init_scale=2.0 ** 16, growth_interval=3)
    sb = torch.amp.GradScaler("cuda", init_scale=2.0 ** 16, growth_interval=3)
    sch_a, sch_b = _schedulers(oa, lr_kind), _schedulers(ob, lr_kind)
    gen = torch.Generator(device=DEV).manual_seed(3)
    scales = {}
    for it in range(1, 13):
        grads = [torch.randn(p.shape, device=DEV, generator=gen) * (1e-2 if it % 3 else 1.0) for p in pa]
        if it in INJECT:
            grads[20].view(-1)[123] = INJECT[it]
        for ps, sc in ((pa, sa), (pb, sb)):
            for p, g in zip(ps, sc.scale(grads)):
                p.grad = g
        before = _state(ob, pb) if it in INJECT else None
        scale_before = sb.get_scale()

        sa.unscale_(oa)
        norm_a = torch.nn.utils.clip_grad_norm_(pa, 1.0)
        sa.step(oa)
        sa.update()
        if order == "train_py":
            sb.unscale_(ob)
            norm_b = torch.nn.utils.clip_grad_norm_(pb, 1.0)
            sb.step(ob)
        else:
            norm_b = sb.step(ob, clip_max_norm=1.0)
        sb.update()
        _sched_step(sch_a, it)
        _sched_step(sch_b, it)
        torch.cuda.synchronize()

        scales[it] = sb.get_scale()
        assert scales[it] == sa.get_scale(), (it, scales[it], sa.get_scale())
        if it in INJECT:
            after = _state(ob, pb)
            changed = [i for i, (x, y) in enumerate(zip(before, after)) if not torch.equal(x, y)]
            assert not changed, f"step {it} ({INJECT[it]}): tensors changed by a skipped step: {changed[:8]}"
            assert scales[it] == scale_before / 2, (it, scale_before, scales[it])
        else:
            e = abs(float(norm_b) - float(norm_a)) / float(norm_a)
            assert e <= OPT_TOL, f"step {it}: total norm {float(norm_b)} vs torch {float(norm_a)}"
            if order == "folded":          # p.grad holds the unscaled, clipped gradient, as after unscale_ + clip
                eg = max(_maxrel(b.grad, a.grad) for a, b in zip(pa, pb))
                assert eg <= OPT_TOL, f"step {it}: clipped gradient max-rel {eg:.3e}"
        lr_a, lr_b_now = oa.param_groups[0]["lr"], float(ob.param_groups[0]["lr"])
        assert abs(lr_b_now - lr_a) <= 1e-6 * lr_a, (it, lr_b_now, lr_a)
    assert scales[7] == 2 * scales[4], scales          # 3 clean steps after the inf: the scale grows again
    for name, get in (("w", lambda o, p: p), ("square_avg", lambda o, p: o.state[p]["square_avg"]),
                      ("momentum_buffer", lambda o, p: o.state[p]["momentum_buffer"])):
        worst = max((_maxrel(get(ob, b), get(oa, a)), i) for i, (a, b) in enumerate(zip(pa, pb)))
        assert worst[0] <= OPT_TOL, f"{name} of tensor {worst[1]}: max-rel {worst[0]:.3e}"
    for a, b in zip(pa, pb):
        assert float(ob.state[b]["step"]) == float(oa.state[a]["step"]) == 12 - len(INJECT)
    if lr_kind == "plateau":
        assert float(ob.param_groups[0]["lr"]) < 1e-4     # the schedule did move


@pytest.mark.gpu
def test_direct_step_with_grad_scale():
    """opt.step() with only grad_scale set (no GradScaler): the norm pass computes found_inf itself."""
    from unetb200.optim import FusedRMSprop
    ws = _unet_weights()[:6]
    pa = [torch.nn.Parameter(w.to(DEV)) for w in ws]
    pb = [torch.nn.Parameter(w.to(DEV)) for w in ws]
    oa = FusedRMSprop(pa, lr=1e-3, momentum=0.9)
    ob = FusedRMSprop(pb, lr=1e-3, momentum=0.9)
    gen = torch.Generator(device=DEV).manual_seed(5)
    for it, bad in enumerate((None, float("inf"), None, float("nan"), None)):
        grads = [torch.randn(p.shape, device=DEV, generator=gen) for p in pa]
        if bad is not None:
            grads[2].view(-1)[0] = bad
        before = _state(ob, pb) if it else None
        for a, b, g in zip(pa, pb, grads):
            a.grad = g.clone()
            b.grad = g * 8.0
        clip = 0.5 if it in (0, 1, 4) else None
        ob.grad_scale = torch.full((), 8.0, device=DEV)
        ob.step(clip_max_norm=clip)
        del ob.grad_scale
        if bad is None:
            oa.step(clip_max_norm=clip)
        else:
            after = _state(ob, pb)
            assert all(torch.equal(x, y) for x, y in zip(before, after)), f"step {it}: a {bad} gradient moved state"
        torch.cuda.synchronize()
    for a, b in zip(pa, pb):
        assert _maxrel(b, a) <= OPT_TOL
        assert _maxrel(ob.state[b]["momentum_buffer"], oa.state[a]["momentum_buffer"]) <= OPT_TOL
        assert float(ob.state[b]["step"]) == float(oa.state[a]["step"]) == 3


@pytest.mark.gpu
@pytest.mark.parametrize("lr_kind", ["tensor", "float"])
def test_folded_step_does_not_sync(lr_kind):
    from unetb200.optim import FusedRMSprop
    ws = _unet_weights()
    ps = [torch.nn.Parameter(w.to(DEV)) for w in ws]
    lr = torch.tensor(1e-3, device=DEV) if lr_kind == "tensor" else 1e-3
    opt = FusedRMSprop(ps, lr=lr, weight_decay=1e-8, momentum=0.999)
    scaler = torch.amp.GradScaler("cuda")
    gen = torch.Generator(device=DEV).manual_seed(1)
    sets = [[torch.randn(p.shape, device=DEV, generator=gen) for p in ps] for _ in range(2)]
    for grads in sets:
        for p, g in zip(ps, scaler.scale(grads)):
            p.grad = g
        torch.cuda.synchronize()
        if grads is sets[1]:                     # the first step creates the scaler's and optimizer's state
            torch.cuda.set_sync_debug_mode("error")
        try:
            scaler.step(opt, clip_max_norm=1.0)
            scaler.update()
        finally:
            torch.cuda.set_sync_debug_mode(0)
    torch.cuda.synchronize()
    assert all(float(opt.state[p]["step"]) == 2 for p in ps)


# ------------------------------------------------------------------------------------------------
# GPU, end to end
# ------------------------------------------------------------------------------------------------
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _model(cls_name, n_classes, state):
    import unet.unet_model as UM
    from unetb200 import functional as UF
    UF._PRE.clear()
    UF._EVAL_COEFS.clear()
    m = getattr(UM, cls_name)(1, n_classes)
    m.load_state_dict(state)
    return m.to(DEV).to(memory_format=torch.channels_last).train()


def _trainer(m):
    """train.py's step with the library's criterion: bf16 autocast, GradScaler, FusedRMSprop with a tensor lr under
    CosineAnnealingWarmRestarts, clip folded into scaler.step."""
    from unetb200 import losses as UL
    from unetb200.optim import FusedRMSprop
    opt = FusedRMSprop(m.parameters(), lr=torch.tensor(1e-3, device=DEV), weight_decay=1e-8, momentum=0.999)
    sched = torch.optim.lr_scheduler.CosineAnnealingWarmRestarts(opt, T_0=3)
    scaler = torch.amp.GradScaler("cuda", init_scale=2.0 ** 12)

    def scaled_loss(x, t):
        with torch.autocast("cuda", dtype=torch.bfloat16):
            loss = UL.training_criterion(m(x), t)
        return scaler.scale(loss)

    def opt_step():
        scaler.step(opt, clip_max_norm=1.0)
        scaler.update()

    def step(x, t):
        for p in m.parameters():
            p.grad = None
        sl = scaled_loss(x, t)
        sl.backward()
        opt_step()
        return sl
    return opt, sched, scaler, scaled_loss, opt_step, step


@pytest.mark.gpu
@pytest.mark.parametrize("cls_name,n_classes,kind", [("UNet_S", 3, "graphed"), ("UNet", 2, "graphed"),
                                                     ("UNet", 2, "segmented")])
def test_captured_amp_step_matches_eager(cls_name, n_classes, kind, monkeypatch):
    """Six replays (scheduler.step() between them) against six eager steps of the same code, B = 2, 96x80; the
    fourth batch has a NaN pixel: its replay leaves the weights unchanged and halves the scale."""
    import unet.unet_model as UM
    from oracle import unet_oracle as O
    from unetb200 import ddp
    from unetb200.graph import GraphedStep
    monkeypatch.setenv("UNET_B200_PRECISION", "fp32")
    if kind == "segmented":
        monkeypatch.setenv("MASTER_ADDR", "127.0.0.1")
        monkeypatch.setenv("MASTER_PORT", str(_free_port()))
        dist.init_process_group("gloo", rank=0, world_size=1)
    torch.manual_seed(7)
    state = {k: v.detach().clone() for k, v in getattr(UM, cls_name)(1, n_classes).state_dict().items()}
    batches = []
    for i in range(7):
        img, msk = O.synthetic_batch(2, 1, n_classes, 96, 80, rank=i)
        if i == 4:
            img[1, 0, 40, 33] = float("nan")
        batches.append((img.to(DEV).contiguous(memory_format=torch.channels_last), msk.to(DEV)))
    nan_step = 4

    def run(captured):
        m = _model(cls_name, n_classes, state)
        opt, sched, scaler, scaled_loss, opt_step, step = _trainer(m)
        if not captured:
            for _ in range(2):                         # the warm-up steps of the captured run
                step(*batches[0])
            go = step
        elif kind == "graphed":
            g = GraphedStep(step, batches[0], warmup=2)
            go = g
        else:
            g = ddp.SegmentedStep(m, scaled_loss, opt_step, batches[0], warmup=2)
            go = g
        rec = []
        try:
            for i in range(1, 7):
                w0 = [p.detach().clone() for p in m.parameters()] if i == nan_step else None
                s0 = scaler.get_scale()
                loss = float(go(*batches[i]).detach())
                torch.cuda.synchronize()
                if w0 is not None:
                    moved = [k for k, (p, w) in enumerate(zip(m.parameters(), w0)) if not torch.equal(p.detach(), w)]
                    assert not moved, f"{kind}: the NaN batch moved parameters {moved[:8]}"
                    assert scaler.get_scale() == s0 / 2, (kind, s0, scaler.get_scale())
                else:
                    assert math.isfinite(loss), (i, loss)
                sched.step()
                lr = float(opt.param_groups[0]["lr"])
                assert lr == float(sched.get_last_lr()[0]), (i, lr, sched.get_last_lr())
                rec.append((loss, lr, scaler.get_scale()))
            weights = {k: p.detach().clone() for k, p in m.named_parameters()}
        finally:
            if captured and kind == "segmented":
                g.release()
        return rec, weights

    try:
        eager, w_eager = run(False)
        replay, w_replay = run(True)
    finally:
        if kind == "segmented":
            dist.destroy_process_group()
    for i, ((le, lre, se), (lr_, lrr, sr)) in enumerate(zip(eager, replay), start=1):
        assert lrr == lre and sr == se, (i, eager, replay)
        if i != nan_step:
            assert abs(lr_ - le) <= GRAPH_TOL * abs(le), (i, eager, replay)
    assert len({lr for _, lr, _ in eager}) >= 3, "the schedule should move the LR"
    worst = max((_maxrel(w_replay[k], w_eager[k]), k) for k in w_eager)
    assert worst[0] <= GRAPH_TOL, f"{kind} {cls_name}: {worst[1]} differs from eager by {worst[0]:.3e} (max-rel)"
