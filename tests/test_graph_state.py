"""State the library keeps outside autograd's view, exercised the way training loops use it.

The library caches packed weight operands (functional._PRE) and eval-mode BatchNorm coefficients
(functional._EVAL_COEFS), lets kernels write gradients straight into registered sinks, and batches the split
reductions of weight gradients (ops._REDUCE_JOBS).  These tests drive a model through several modes in a row --
CUDA-graph replays then evaluation, replays then an eager step, SegmentedStep on every model variant, a backward
pass that raises and its retry, gradient consumers inside backward -- and compare each result with a fresh model or
with a plain PyTorch-CPU fp32 restatement of the same operation.  The last test checks the reduction queue on the CPU.
"""
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.nn.functional as F

DEV = "cuda"
MODES = ("fp32", "bf16")
INFER_TOL = {"fp32": (1e-3, 1e-3), "bf16": (1e-1, 2e-2)}      # (logits max-rel, argmax mismatch): infer_gate's bars


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


@pytest.fixture
def gloo_world1():
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(_free_port())
    dist.init_process_group("gloo", rank=0, world_size=1)
    try:
        yield
    finally:
        dist.destroy_process_group()


@pytest.fixture
def precision(request, monkeypatch):
    """'fp32': exact CUDA-core arithmetic, no autocast; 'bf16': autocast (the tcgen05 kernels)."""
    monkeypatch.setenv("UNET_B200_PRECISION", "fp32")
    return request.param


@pytest.fixture
def clean_queues():
    """Host-side reset of the reduction queue and side-stream bookkeeping after a test, so that a failure in one test
    can never leave work behind that a later backward pass would launch."""
    yield
    from unetb200 import ops
    torch.cuda.synchronize()
    ops._REDUCE_JOBS.clear()
    ops._REDUCE_PENDING[0] = None
    ops._SIDE_KEEP.clear()
    ops._SIDE_PENDING[0] = False


def _ctx(mode):
    return torch.autocast("cuda", enabled=(mode == "bf16"))


def _host(t):
    return t.detach().float().cpu()


def _batch(B=2, H=64, W=64):
    from oracle import unet_oracle as O
    img, msk = O.synthetic_batch(B, 1, 2, H, W)
    return img, img.to(DEV).contiguous(memory_format=torch.channels_last), msk.to(DEV)


def _fresh(state, cls=None, channels_last=True):
    """A new model that loaded `state` with both caches emptied first."""
    import unet
    from unetb200 import functional as UF
    UF._PRE.clear()
    UF._EVAL_COEFS.clear()
    m = (cls or unet.UNet)(1, 2)
    m.load_state_dict(state)
    m = m.to(DEV)
    if channels_last:
        m = m.to(memory_format=torch.channels_last)
    return m.train()


def _snapshot(m):
    return {k: v.detach().clone() for k, v in m.state_dict().items()}


def _eval_logits(m, x, mode):
    m.eval()
    with torch.inference_mode(), _ctx(mode):
        out = m(x).float().clone()
    m.train()
    return out


def _loss(m, x, t, mode):
    from unetb200 import losses as UL
    with _ctx(mode):
        return UL.training_criterion(m(x), t, boundary_coeff=0.2)


def _maxrel(a, b):
    from oracle import unet_oracle as O
    return O.rel_err(_host(a), _host(b))


# ------------------------------------------------------------------------------------------------
# a. evaluate -> replays -> evaluate
# ------------------------------------------------------------------------------------------------
def _stepper(kind, m, x, t, mode, optimizer):
    """A replayable training step of `m`: (object with .replay(), description)."""
    from unetb200 import ddp
    from unetb200.graph import GraphedStep
    from unetb200.optim import FusedRMSprop
    if optimizer == "none":                 # nothing moves but the BatchNorm running statistics
        ticks = torch.zeros((), device=DEV)
        opt_step = lambda: ticks.add_(1)    # noqa: E731
    elif kind == "graphed_torch_rmsprop":   # INTEGRATION.md section 3
        opt = torch.optim.RMSprop(m.parameters(), lr=1e-4, capturable=True, foreach=True)
        opt_step = opt.step
    else:
        opt = FusedRMSprop(m.parameters(), lr=1e-4)
        opt_step = opt.step
    if kind == "segmented":
        return ddp.SegmentedStep(m, lambda xx, tt: _loss(m, xx, tt, mode), opt_step, (x, t), warmup=2)

    def step(xx, tt):
        for p in m.parameters():
            p.grad = None
        loss = _loss(m, xx, tt, mode)
        loss.backward()
        opt_step()
        return loss
    return GraphedStep(step, (x, t), warmup=2)


@pytest.mark.gpu
@pytest.mark.parametrize("precision", MODES, indirect=True)
@pytest.mark.parametrize("variant", ["weights_and_stats", "weights_only", "stats_only"])
@pytest.mark.parametrize("kind", ["graphed_torch_rmsprop", "graphed_fused_rmsprop", "segmented"])
def test_evaluate_after_replays(precision, variant, kind, gloo_world1):
    """Evaluation between CUDA-graph replays (INTEGRATION.md section 3: train with graph replays, evaluate() every
    epoch) sees the weights and running statistics of the latest replay.  weights_only (BatchNorm momentum 0) isolates
    the packed-operand cache, stats_only (an optimizer that changes nothing) the eval-coefficient cache."""
    from oracle import unet_oracle as O
    mode = precision
    img, x, t = _batch()
    m = _fresh(O.build_state(1, 2, False, seed=0))
    if variant == "weights_only":
        for mod in m.modules():
            if isinstance(mod, torch.nn.BatchNorm2d):
                mod.momentum = 0.0
    step = _stepper(kind, m, x, t, mode, "none" if variant == "stats_only" else "real")
    evals = []
    try:
        for _ in range(2):
            for _ in range(3):
                step.replay()
            evals.append((_eval_logits(m, x, mode), _snapshot(m)))
    finally:
        if kind == "segmented":
            step.release()
    # the fresh models come last: building one empties the caches the evaluations above depended on
    assert not torch.equal(evals[0][1]["inc.double_conv.1.running_mean"], evals[1][1]["inc.double_conv.1.running_mean"]) \
        or not torch.equal(evals[0][1]["inc.double_conv.0.weight"], evals[1][1]["inc.double_conv.0.weight"])
    for k, (ev, state) in enumerate(evals):
        ref = _eval_logits(_fresh(state), x, mode)
        r = O.unet_forward({n: v.cpu() for n, v in state.items()}, img, False, training=False)
        assert torch.equal(ev, ref), (f"evaluation {k + 1} differs from a fresh model's (max-rel {_maxrel(ev, ref):.3e}; "
                                      f"against the CPU oracle: {_maxrel(ev, r):.3e}, fresh {_maxrel(ref, r):.3e})")
        tol, tol_argmax = INFER_TOL[mode]
        assert _maxrel(ev, r) <= tol, f"evaluation {k + 1} against the CPU oracle"
        assert (_host(ev).argmax(1) != r.argmax(1)).float().mean().item() <= tol_argmax


# ------------------------------------------------------------------------------------------------
# b. replays -> an eager step (the partial last batch of an epoch)
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("precision", MODES, indirect=True)
@pytest.mark.parametrize("kind", ["graphed_torch_rmsprop", "graphed_fused_rmsprop"])
def test_eager_step_after_replays(precision, kind):
    from oracle import unet_oracle as O
    mode = precision
    img, x, t = _batch()
    m = _fresh(O.build_state(1, 2, False, seed=0))
    step = _stepper(kind, m, x, t, mode, "real")
    for _ in range(3):
        step.replay()
    torch.cuda.synchronize()
    state = _snapshot(m)
    x1, t1 = x[:1].contiguous(memory_format=torch.channels_last), t[:1].contiguous()
    grads = {}
    for name, model in (("after_replays", m), ("fresh", None)):
        if model is None:
            model = _fresh(state)
        for p in model.parameters():
            p.grad = None
        _loss(model, x1, t1, mode).backward()
        torch.cuda.synchronize()
        grads[name] = {k: _host(p.grad) for k, p in model.named_parameters()}
    a, b = grads["after_replays"], grads["fresh"]
    worst = max(((_maxrel(a[k], b[k]), k) for k in b))
    assert worst[0] <= 1e-6, f"gradient of {worst[1]} differs by {worst[0]:.3e} (max-rel)"


# ------------------------------------------------------------------------------------------------
# c. SegmentedStep produces every parameter's gradient in its bucket view
# ------------------------------------------------------------------------------------------------
def _variant_model(cls_name, channels_last):
    import unet.unet_model as UM
    torch.manual_seed(7)
    st = {k: v.detach().clone() for k, v in getattr(UM, cls_name)(1, 2).state_dict().items()}
    return st, getattr(UM, cls_name)


@pytest.mark.gpu
@pytest.mark.parametrize("cls_name,channels_last", [("UNet_SA", True), ("UNet", False), ("UNet_S", True)])
def test_segmented_step_covers_every_parameter(cls_name, channels_last, monkeypatch):
    from unetb200 import ddp
    from unetb200 import functional as UF
    monkeypatch.setenv("UNET_B200_PRECISION", "fp32")
    st, cls = _variant_model(cls_name, channels_last)
    img, x, t = _batch()
    if not channels_last:
        x = x.contiguous()

    # eager reference: loss.backward() on a fresh model
    ref = _fresh(st, cls, channels_last)
    _loss(ref, x, t, "bf16").backward()
    torch.cuda.synchronize()
    g_ref = {k: _host(p.grad) for k, p in ref.named_parameters()}
    del ref

    m = _fresh(st, cls, channels_last)
    ticks = torch.zeros((), device=DEV)
    step = ddp.SegmentedStep(m, lambda xx, tt: _loss(m, xx, tt, "bf16"), lambda: ticks.add_(1), (x, t), warmup=1)
    try:
        if cls_name == "UNet":
            assert step.grad_copies == 0, "every UNet gradient is written by its kernel into its bucket view"
        step.replay()
        torch.cuda.synchronize()
        views = {id(p): v for b in step.reducer.buckets for p, v in zip(b["params"], b["views"])}
        for k, p in m.named_parameters():
            v = views[id(p)]
            assert p.grad is not None and p.grad.data_ptr() == v.data_ptr() and p.grad.stride() == v.stride(), k
            assert float(p.grad.abs().max()) > 0, f"{k}: zero gradient"
            e = _maxrel(p.grad, g_ref[k])
            assert e <= 1e-6, f"{k}: gradient differs from eager backward by {e:.3e} (max-rel)"
    finally:
        step.release()

    # one replay with an SGD optimizer graph moves every parameter (the attention convolutions included)
    m = _fresh(st, cls, channels_last)
    opt = torch.optim.SGD(m.parameters(), lr=1e-2, foreach=True)
    step = ddp.SegmentedStep(m, lambda xx, tt: _loss(m, xx, tt, "bf16"), opt.step, (x, t), warmup=1)
    try:
        before = {k: p.detach().clone() for k, p in m.named_parameters()}
        step.replay()
        torch.cuda.synchronize()
        still = [k for k, p in m.named_parameters() if torch.equal(p.detach(), before[k])]
        assert not still, f"parameters the SGD replay did not move: {still}"
        if cls_name == "UNet_SA":
            assert all(f"{u}.attention.conv1.weight" not in still for u in ("up1", "up2", "up3", "up4"))
    finally:
        step.release()
    assert not UF._GRAD_SINK


# ------------------------------------------------------------------------------------------------
# d. a backward pass that raises, then the retry with activation re-computation (train.py's OOM path)
# ------------------------------------------------------------------------------------------------
class _Boom(RuntimeError):
    pass


@pytest.mark.gpu
@pytest.mark.parametrize("wgrad_side", [False, True])
def test_failed_backward_then_retry(wgrad_side, monkeypatch, clean_queues):
    from oracle import unet_oracle as O
    from unetb200 import ops
    monkeypatch.setenv("UNET_B200_PRECISION", "fp32")
    monkeypatch.setattr(ops, "_WGRAD_SIDE", wgrad_side)
    st = O.build_state(1, 2, False, seed=0)
    img, x, t = _batch()
    m = _fresh(st)
    run = m.inc.run

    def boom(g):
        raise _Boom("backward failed")

    def failing_run(*a, **k):
        out = run(*a, **k)
        out[0].register_hook(boom)
        return out
    m.inc.run = failing_run
    loss = _loss(m, x, t, "bf16")
    with pytest.raises(_Boom):
        loss.backward()          # inc's backward runs last: the other stages' weight gradients are done by now
    del m.inc.run, loss
    _loss(m, x, t, "bf16")       # a forward only: its graph is dropped at once
    assert not ops._REDUCE_JOBS, "reductions of the failed pass are still queued"
    assert not ops._SIDE_KEEP, "operands of the failed pass are still held for the side stream"

    m.use_checkpointing()
    for p in m.parameters():
        p.grad = None
    _loss(m, x, t, "bf16").backward()
    torch.cuda.synchronize()

    ref = _fresh(st)
    for _ in range(2):           # the failed pass's and the lone forward's statistics updates
        _loss(ref, x, t, "bf16")
    _loss(ref, x, t, "bf16").backward()
    torch.cuda.synchronize()
    g = {k: _host(p.grad) for k, p in ref.named_parameters()}
    for k, p in m.named_parameters():
        assert _maxrel(p.grad, g[k]) <= 1e-6, k
    s_ref = ref.state_dict()
    for k, v in m.state_dict().items():
        if "running" in k:
            assert _maxrel(v, s_ref[k]) <= 1e-6, k
        elif "tracked" in k:
            assert int(v) == int(s_ref[k]) == 3, k


# ------------------------------------------------------------------------------------------------
# e. gradient consumers inside backward
# ------------------------------------------------------------------------------------------------
def _grads_with_consumers(build, run, defer, monkeypatch):
    from unetb200 import ops
    monkeypatch.setattr(ops, "DEFER_REDUCE", defer)
    model = build()
    out = run(model)
    torch.cuda.synchronize()
    return model, out


@pytest.mark.gpu
def test_accumulate_grad_prehooks_see_final_gradients(monkeypatch):
    """A pre-hook on the AccumulateGrad node (where DistributedDataParallel and FSDP attach) reads each gradient as
    autograd hands it over: it must already be complete."""
    from oracle import unet_oracle as O
    monkeypatch.setenv("UNET_B200_PRECISION", "fp32")
    st = O.build_state(1, 2, False, seed=0)
    img, x, t = _batch()
    res = {}
    for defer in (True, False):
        def run(m):
            seen, nodes, handles = {}, [], []
            for k, p in m.named_parameters():
                node = torch.autograd.graph.get_gradient_edge(p).node
                nodes.append(node)

                def hook(grads, k=k):
                    seen[k] = grads[0].detach().clone()
                handles.append(node.register_prehook(hook))
            _loss(m, x, t, "bf16").backward()
            for h in handles:
                h.remove()
            return seen
        m, seen = _grads_with_consumers(lambda: _fresh(st), run, defer, monkeypatch)
        for k, p in m.named_parameters():
            assert _maxrel(seen[k], p.grad) <= 1e-6, f"{k}: the hook saw an unfinished gradient (defer={defer})"
        res[defer] = {k: _host(p.grad) for k, p in m.named_parameters()}
    for k in res[False]:
        assert _maxrel(res[True][k], res[False][k]) <= 1e-6, k


def _cpu_double_conv(x, w1, g1, b1, w2, g2, b2):
    """conv3x3 (no bias) -> training BatchNorm -> ReLU, twice: PyTorch-CPU fp32."""
    for w, g, b in ((w1, g1, b1), (w2, g2, b2)):
        x = F.relu(F.batch_norm(F.conv2d(x, w, padding=1), None, None, g, b, training=True, eps=1e-5))
    return x


@pytest.mark.gpu
def test_shared_module_used_twice(monkeypatch):
    """One DoubleConv applied twice in a forward pass: autograd sums the two contributions to each weight gradient
    before AccumulateGrad."""
    from unet import unet_parts as P
    monkeypatch.setenv("UNET_B200_PRECISION", "fp32")
    torch.manual_seed(11)
    dc = P.DoubleConv(32, 32)
    with torch.no_grad():
        for bn in (dc.double_conv[1], dc.double_conv[4]):
            bn.weight.uniform_(0.5, 1.5)
            bn.bias.uniform_(-0.2, 0.2)
    st = {k: v.clone() for k, v in dc.state_dict().items()}
    g = torch.Generator().manual_seed(12)
    x_h = torch.randn(2, 32, 24, 20, generator=g)
    gout = torch.randn(2, 32, 24, 20, generator=g)

    class Twice(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.dc = P.DoubleConv(32, 32)

        def forward(self, x):
            return self.dc(self.dc(x))

    res = {}
    for defer in (True, False):
        def build():
            m = Twice()
            m.dc.load_state_dict(st)
            return m.to(DEV).to(memory_format=torch.channels_last).train()

        def run(m):
            x = x_h.to(DEV).contiguous(memory_format=torch.channels_last).requires_grad_(True)
            y = m(x)
            y.backward(gout.to(DEV))
            return _host(y), _host(x.grad)
        m, (y, gx) = _grads_with_consumers(build, run, defer, monkeypatch)
        res[defer] = (y, gx, {k: _host(p.grad) for k, p in m.dc.named_parameters()})
    for k in res[False][2]:
        assert _maxrel(res[True][2][k], res[False][2][k]) <= 1e-6, k

    ps = {k: v.clone().requires_grad_(True) for k, v in st.items() if "running" not in k and "tracked" not in k}
    order = [ps[f"double_conv.{i}.{n}"] for i, n in ((0, "weight"), (1, "weight"), (1, "bias"), (3, "weight"),
                                                     (4, "weight"), (4, "bias"))]
    x_r = x_h.clone().requires_grad_(True)
    y_r = _cpu_double_conv(_cpu_double_conv(x_r, *order), *order)
    y_r.backward(gout)
    y, gx, gp = res[True]
    assert _maxrel(y, y_r) <= 2e-4
    assert _maxrel(gx, x_r.grad) <= 2e-4
    for k, p in ps.items():
        assert _maxrel(gp[k], p.grad) <= 2e-4, k


@pytest.mark.gpu
def test_stock_ddp_world1(gloo_world1, monkeypatch):
    from oracle import unet_oracle as O
    try:
        probe = torch.ones(1, device=DEV)
        dist.all_reduce(probe)
        torch.cuda.synchronize()
    except Exception as exc:  # noqa: BLE001
        pytest.skip(f"this build's gloo cannot all-reduce CUDA tensors: {exc}")
    monkeypatch.setenv("UNET_B200_PRECISION", "fp32")
    st = O.build_state(1, 2, False, seed=0)
    img, x, t = _batch()
    res = {}
    for defer in (True, False):
        def run(m):
            d = torch.nn.parallel.DistributedDataParallel(m, device_ids=[0])
            _loss(d, x, t, "bf16").backward()
            return d
        m, _ = _grads_with_consumers(lambda: _fresh(st), run, defer, monkeypatch)
        res[defer] = {k: _host(p.grad) for k, p in m.named_parameters()}
    for k in res[False]:
        assert _maxrel(res[True][k], res[False][k]) <= 1e-6, k


# ------------------------------------------------------------------------------------------------
# f. the reduction queue on the CPU: nothing of an aborted pass reaches the next pass's flush
# ------------------------------------------------------------------------------------------------
def test_reduce_queue_drops_jobs_of_a_failed_pass(monkeypatch):
    from unetb200 import ops
    flushed = []

    def record():
        flushed.append([j[1] for j in ops._REDUCE_JOBS])
        ops._REDUCE_JOBS.clear()
        ops._REDUCE_PENDING[0] = None
    monkeypatch.setattr(ops, "_REDUCE_JOBS", [])
    monkeypatch.setattr(ops, "_REDUCE_PENDING", [None])
    monkeypatch.setattr(ops, "flush_wgrad_reduce", record)

    def job(dst):
        return (torch.zeros(4), dst, 1, 1, 0, 1, 2, 1, 1, 1, 1)

    class Queue(torch.autograd.Function):
        @staticmethod
        def forward(ctx, x, dst, fail):
            ctx.dst, ctx.fail = dst, fail
            return x * 2

        @staticmethod
        def backward(ctx, g):
            ops._queue_reduce(job(ctx.dst))
            if ctx.fail:
                raise _Boom("backward failed")
            return g * 2, None, None

    x = torch.ones(3, requires_grad=True)
    with pytest.raises(_Boom):
        Queue.apply(x, 0x1000, True).sum().backward()
    assert flushed == []
    Queue.apply(x, 0x2000, False).sum().backward()
    assert flushed == [[0x2000]], f"the flush saw {flushed}"
    # outside any backward pass a job is reduced at once
    ops._queue_reduce(job(0x3000))
    assert flushed[-1] == [0x3000]
