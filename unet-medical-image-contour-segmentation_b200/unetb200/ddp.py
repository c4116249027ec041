"""Data-parallel gradient exchange for the UNet step (BASELINE.json configs[3]).

The reference is single-device (train.py:244); this layer has no counterpart there.  Semantics are
standard DDP: replicated weights (broadcast from rank 0), per-replica BatchNorm batch statistics (the
reference uses plain nn.BatchNorm2d), gradients mean-reduced over ranks.  The only exchange step of
the path is that all-reduce, so it is the only collective: NCCL over NVLink 5 / NVSwitch through
torch.distributed.

Two ways to drive it:

* :class:`GradAllReducer` -- eager launches: ``loss.backward(); reducer.finish()``.  Buckets are all-reduced from
  autograd hooks while backward is still running (buckets fill in reverse layer order: outc, up4 ... inc), on
  NCCL's own stream, joined once before the optimizer step.  The backward kernels write every gradient straight
  into its bucket (``functional.set_grad_sinks``), so there is no packing copy.
* :class:`SegmentedStep` -- CUDA graphs: the forward pass, the backward pass cut into four segments at
  activations of the network, and the optimizer step are captured as separate graphs that share one memory pool;
  between two backward segments the bucket the finished segment has filled is all-reduced eagerly on NCCL's
  stream while the next segment's graph runs.  Only the last bucket (down2 / down1 / inc: 1.1 M values) is
  exposed.  (A single graph holding the NCCL calls hangs on this stack, and one graph for the whole backward
  pass leaves the 124 MB all-reduce fully exposed: DESIGN.md section 5.)

Works with the gloo backend on CPU tensors too (used by the CPU tests).
"""
from __future__ import annotations

import torch
import torch.distributed as dist

from . import backward_pass


def _functional():
    try:
        from . import functional
        return functional
    except Exception:  # noqa: BLE001  (CPU-only use of this module in the gloo tests: no library, no sinks)
        return None


def broadcast_module_state(module, src=0):
    """Replicate parameters and buffers from `src` (rank-0 convention for BN running stats)."""
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return
    with torch.no_grad():
        for t in list(module.parameters()) + list(module.buffers()):
            dist.broadcast(t.data, src=src)


def sync_buffers(module, src=0):
    """BatchNorm running statistics are per replica during training (like a per-GPU nn.BatchNorm2d); before a
    checkpoint or an evaluation pass that should not depend on the rank, replicate `src`'s buffers."""
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return
    with torch.no_grad():
        for t in module.buffers():
            dist.broadcast(t.data, src=src)


# ------------------------------------------------------------------------------------------------
# synchronised BatchNorm (nn.SyncBatchNorm holders): statistics exchanged over NVLink by kernel stores
# ------------------------------------------------------------------------------------------------
SYNC_BN_MAX_CHANNELS = 4096        # exchange-buffer capacity per layer (UNet's widest layer has 1024 channels)
_PEER_GROUPS = {}                  # (device index, process group) -> BNPeerGroup


def sync_bn_process_group(module, training=False):
    """(number of nn.SyncBatchNorm layers in `module`, the process group they name: None = WORLD).  Raises ValueError
    when they name different groups (one peer group serves a model), and for training when one of them has
    momentum=None (as the forward pass of such a layer does)."""
    layers = [m for m in module.modules() if isinstance(m, torch.nn.SyncBatchNorm)]
    groups = {id(m.process_group): m.process_group for m in layers}
    if len(groups) > 1:
        raise ValueError("unetb200: the SyncBatchNorm layers of one model must all name the same process group")
    if training and any(m.momentum is None for m in layers):
        raise ValueError("unetb200: SyncBatchNorm(momentum=None) (cumulative average) is not supported")
    return len(layers), (next(iter(groups.values())) if groups else None)


def bn_sync_group(bn, device):
    """The BNPeerGroup a training-mode BatchNorm holder synchronises over, or None when it normalises with its own
    batch: not an nn.SyncBatchNorm, torch.distributed not initialised, or a group of one rank (torch's rule).
    Creates the peer group on first use (a collective of the group: every rank's first synchronised forward)."""
    if not isinstance(bn, torch.nn.SyncBatchNorm) or not (dist.is_available() and dist.is_initialized()):
        return None
    group = bn.process_group if bn.process_group is not None else dist.group.WORLD
    key = (device.index, group)
    pg = _PEER_GROUPS.get(key)
    if pg is not None:
        return pg
    if dist.get_world_size(group) <= 1:
        return None
    if torch.cuda.is_current_stream_capturing():
        raise RuntimeError("unetb200: the first synchronised BatchNorm forward must run eagerly (it sets up the "
                           "NVLink peer group, a collective): run one step before capturing a CUDA graph "
                           "(SegmentedStep's warm-up does)")
    pg = _PEER_GROUPS[key] = BNPeerGroup(group, device)
    return pg


class BNPeerGroup:
    """The ranks of one process group on one device, with their mapped exchange buffers (libunetb200's
    unetb200_bn_peer_group_t).  Created by bn_sync_group, torn down by destroy_peer_groups."""

    def __init__(self, group, device, max_channels=SYNC_BN_MAX_CHANNELS):
        import ctypes as C

        from . import _lib
        L = _lib.load()
        self.group, self.device = group, device
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)
        handle, bus = C.create_string_buffer(64), C.create_string_buffer(32)
        h = C.c_void_p()
        with torch.cuda.device(device):
            _lib.check(L.unetb200_bn_peer_group_create(self.rank, self.world, max_channels, handle, bus, C.byref(h)),
                       "bn_peer_group_create")
            self.handle = h
            try:
                parts = [None] * self.world
                dist.all_gather_object(parts, (handle.raw, bus.raw), group=group)
                rc = L.unetb200_bn_peer_group_open(h, b"".join(p[0] for p in parts), b"".join(p[1] for p in parts))
                msg = L.unetb200_last_error().decode("utf-8", "replace") if rc else ""
                status = [None] * self.world           # every rank learns whether every rank could map its peers
                dist.all_gather_object(status, (rc, msg), group=group)
            except BaseException:
                L.unetb200_bn_peer_group_destroy(h)
                raise
        bad = [f"rank {r}: {m}" for r, (rc, m) in enumerate(status) if rc != 0]
        if bad:
            L.unetb200_bn_peer_group_destroy(h)
            self.handle = None
            raise RuntimeError("unetb200: SyncBatchNorm needs every pair of ranks to reach each other by CUDA peer "
                               "access (one node): " + "; ".join(bad))

    def check(self):
        """Raise if an exchange of this group has timed out (a rank stopped taking part)."""
        import ctypes as C

        from . import _lib
        if self.handle is None:
            raise RuntimeError("unetb200: SyncBatchNorm peer group used after destroy_peer_groups()")
        missing, epoch = C.c_int64(), C.c_int64()
        _lib.check(_lib.load().unetb200_bn_peer_group_status(self.handle, C.byref(missing), C.byref(epoch)),
                   "bn_peer_group_status")
        if missing.value >= 0:
            raise RuntimeError(f"unetb200: SyncBatchNorm exchange {epoch.value} on rank {self.rank} timed out waiting "
                               f"for rank {missing.value}; the peer group is unusable (destroy_peer_groups())")

    def destroy(self):
        from . import _lib
        if self.handle is None:
            return
        with torch.cuda.device(self.device):
            torch.cuda.synchronize()
            if dist.is_initialized():
                dist.barrier(group=self.group)          # no rank still writes into this rank's buffer
            _lib.load().unetb200_bn_peer_group_destroy(self.handle)
        self.handle = None


def destroy_peer_groups():
    """Tear down every SyncBatchNorm peer group of this process: a collective of each group, to be called by every
    rank before dist.destroy_process_group()."""
    for key in list(_PEER_GROUPS):
        _PEER_GROUPS.pop(key).destroy()


def check_peer_groups():
    """Raise if an exchange of any SyncBatchNorm peer group has timed out (for graph replays, which have no Python
    entry per exchange)."""
    for pg in _PEER_GROUPS.values():
        pg.check()


class GradAllReducer:
    """Bucketed, backward-overlapped mean all-reduce of ``module``'s gradients.

    Usage per step:  ``loss.backward(); reducer.finish()``  (then clip / optimizer.step()).
    After ``finish()`` every ``p.grad`` is a view into its bucket holding the rank-averaged gradient.
    One backward pass per ``finish()``: gradient accumulation over several backward passes is not supported and
    raises (a second pass would add into a bucket that is already being reduced).
    """

    def __init__(self, module, bucket_bytes=32 << 20, group=None, overlap=None, groups=None, sinks=True,
                 sinks_always=False):
        # overlap=True launches each bucket's all-reduce from the autograd hook that completes it (while backward
        # is still running); overlap=False launches them all from finish().  Default: UNETB200_DDP_OVERLAP, else on.
        if overlap is None:
            import os
            overlap = os.environ.get("UNETB200_DDP_OVERLAP", "1") != "0"
        self.overlap = bool(overlap)
        self.manual = False          # True: hooks are inert, the caller drives launch_bucket / wait_all
        self.group = group
        self.world = dist.get_world_size(group) if (dist.is_available() and dist.is_initialized()) else 1
        self.params = [p for p in module.parameters() if p.requires_grad]
        self.buckets = []          # list of dict(params, offsets, numel, buffer, pending, work, views)
        if groups is not None:     # explicit buckets (SegmentedStep: one per backward segment)
            seen = set()
            for g in groups:
                g = [p for p in g if p.requires_grad]
                seen.update(id(p) for p in g)
                if g:
                    self._close_bucket(g)
            missing = [p for p in self.params if id(p) not in seen]
            if missing:
                raise ValueError("GradAllReducer: `groups` must cover every parameter that requires a gradient")
        else:
            # reverse registration order ~ order in which backward produces the gradients
            cur, cur_bytes = [], 0
            for p in reversed(self.params):
                nbytes = p.numel() * 4
                if cur and cur_bytes + nbytes > bucket_bytes:
                    self._close_bucket(cur)
                    cur, cur_bytes = [], 0
                cur.append(p)
                cur_bytes += nbytes
            if cur:
                self._close_bucket(cur)
        self._where = {}
        for bi, b in enumerate(self.buckets):
            for pi, p in enumerate(b["params"]):
                self._where[p] = (bi, pi)
        self._handles = [p.register_post_accumulate_grad_hook(self._on_grad) for p in self.params]
        self.launched = 0
        self._sinks = False
        F = _functional() if sinks else None
        if F is not None and all(p.is_cuda for p in self.params):
            for b in self.buckets:
                F.set_grad_sinks(b["params"], b["views"], always=sinks_always)
            self._sinks = True

    def _close_bucket(self, params):
        offsets, n = [], 0
        for p in params:
            offsets.append(n)
            n += (p.numel() + 3) // 4 * 4          # every view 16-byte aligned (vector loads of the optimizer)
        dev = params[0].device
        b = dict(params=list(params), offsets=offsets, numel=n,
                 buffer=torch.zeros(n, dtype=torch.float32, device=dev), pending=len(params), work=None)
        b["views"] = self._views(b)
        self.buckets.append(b)

    def _views(self, b):
        """Bucket slices shaped AND strided like their parameters (a channels_last parameter gets a channels_last
        gradient view), so that optimizers and AccumulateGrad see the layout they expect and nothing re-copies."""
        out = []
        for p, o in zip(b["params"], b["offsets"]):
            flat = b["buffer"][o:o + p.numel()]
            dense = sorted((st, sz) for sz, st in zip(p.shape, p.stride()) if sz > 1)
            expect, ok = 1, True
            for st, sz in dense:
                ok = ok and st == expect
                expect *= sz
            out.append(flat.as_strided(p.shape, p.stride()) if ok and p.dim() > 0 else flat.view_as(p))
        return out

    def _fill(self, b):
        """Bring every gradient of bucket `b` into the bucket (no-op for those a backward kernel wrote there)."""
        src, dst = [], []
        for p, v in zip(b["params"], b["views"]):
            g = p.grad
            if g is None:
                v.zero_()
            elif g.data_ptr() != v.data_ptr() or g.stride() != v.stride() or g.dtype != torch.float32:
                src.append(g.to(torch.float32))
                dst.append(v)
        if src:
            torch._foreach_copy_(dst, src)

    def _allreduce(self, b):
        if dist.get_backend(self.group) == "nccl":       # NCCL averages inside the collective
            return dist.all_reduce(b["buffer"], op=dist.ReduceOp.AVG, group=self.group, async_op=True)
        b["buffer"].mul_(1.0 / self.world)
        return dist.all_reduce(b["buffer"], op=dist.ReduceOp.SUM, group=self.group, async_op=True)

    # ---- explicit form (used when the step is replayed as CUDA graphs: the collective stays outside the captured
    # regions) -- fill inside the graphs (or nothing to fill: sinks), launch_bucket eagerly, wait_all before the
    # optimizer graph
    def pack_all(self):
        """Bring every gradient into its bucket (no communication)."""
        backward_pass.side_stream_sync()
        for b in self.buckets:
            self._fill(b)

    def launch_bucket(self, i):
        """Start the mean all-reduce of bucket i on NCCL's stream, ordered after the current stream."""
        if self.world == 1:
            return
        b = self.buckets[i]
        b["work"] = self._allreduce(b)
        self.launched += 1

    def wait_all(self):
        """Order the current stream after every outstanding all-reduce."""
        for b in self.buckets:
            if b["work"] is not None:
                b["work"].wait()
                b["work"] = None

    def allreduce_all(self):
        """Mean all-reduce of every bucket; returns when the results are ordered on the current stream."""
        if self.world == 1:
            return
        for i in range(len(self.buckets)):
            self.launch_bucket(i)
        self.wait_all()

    def point_grads(self):
        """p.grad = its (averaged) bucket view."""
        for b in self.buckets:
            for p, v in zip(b["params"], b["views"]):
                p.grad = v

    def _on_grad(self, p):
        if self.world == 1 or self.manual:
            return
        bi, _ = self._where[p]
        b = self.buckets[bi]
        if b["work"] is not None or b["pending"] <= 0:
            raise RuntimeError("GradAllReducer: a gradient arrived for a bucket that is already complete or being "
                               "reduced -- call finish() after every backward pass (gradient accumulation over "
                               "several backward passes is not supported)")
        b["pending"] -= 1
        if b["pending"] == 0 and self.overlap:
            self._launch(b)

    def _launch(self, b):
        backward_pass.side_stream_sync()    # weight gradients may be produced on the library's side stream
        self._fill(b)
        b["work"] = self._allreduce(b)
        self.launched += 1

    def finish(self):
        """Join the outstanding all-reduces and point every p.grad at its averaged bucket view."""
        if self.world == 1:
            return
        for b in self.buckets:
            if b["work"] is None and b["pending"] != len(b["params"]):
                self._launch(b)            # not launched from a hook: overlap off, or parameters without a gradient
        for b in self.buckets:
            if b["work"] is not None:
                b["work"].wait()
                for p, v in zip(b["params"], b["views"]):
                    if p.grad is not None:
                        p.grad = v.to(p.grad.dtype) if p.grad.dtype != torch.float32 else v
                b["work"] = None
            b["pending"] = len(b["params"])

    def remove(self):
        for h in self._handles:
            h.remove()
        self._handles = []
        if self._sinks:
            F = _functional()
            if F is not None:
                F.clear_grad_sinks(self.params)
            self._sinks = False


# ------------------------------------------------------------------------------------------------
# graph-replayed step with the all-reduce hidden behind the backward pass
# ------------------------------------------------------------------------------------------------
# backward segments in execution order: (module names whose parameters the segment produces gradients for)
SEGMENTS = (("outc", "up4", "up3"), ("up2", "up1"), ("down4", "down3"), ("down2", "down1", "inc"))


def segment_params(model):
    return [[p for name in names for p in getattr(model, name).parameters()] for names in SEGMENTS]


def segmented_backward(model, loss, taps, params_by_segment, after_segment=None):
    """The backward pass of `loss` through a unetb200 UNet, run as len(SEGMENTS) torch.autograd.grad calls cut at
    the activations ``model._taps`` recorded during the forward pass (u2 = output of up2; x1..x5 = encoder outputs /
    skips; p3 = pooled output of down2; each as (tensor, cut alias), see functional.CutFn).  Returns the list of per-segment gradient lists (parameter order of
    `params_by_segment`).  after_segment(k): called when segment k's gradients have been enqueued."""
    t = taps
    out = []

    def run(k, outputs, grad_outputs, cut):
        ps = [p for p in params_by_segment[k] if p.requires_grad]
        res = torch.autograd.grad(outputs, ps + cut, grad_outputs, allow_unused=True)
        out.append(list(res[:len(ps)]))
        if after_segment is not None:
            after_segment(k)
        return res[len(ps):]

    src = lambda *names: [t[n][0] for n in names]      # noqa: E731  the tensors themselves (segment outputs)
    cut = lambda *names: [t[n][1] for n in names]      # noqa: E731  their cut aliases (where a segment stops)
    g_u2, g_x2, g_x1 = run(0, [loss], None, cut("u2", "x2", "x1"))
    g_x5, g_x4, g_x3 = run(1, src("u2"), [g_u2], cut("x5", "x4", "x3"))
    (g_p3,) = run(2, src("x5", "x4"), [g_x5, g_x4], cut("p3"))
    run(3, src("x3", "p3", "x2", "x1"), [g_x3, g_p3, g_x2, g_x1], [])
    return out


class SegmentedStep:
    """forward graph | 4 backward-segment graphs with per-segment bucket all-reduces launched in between |
    optimizer graph.  ``fwd_loss(x, t) -> loss`` runs the model and the criterion; ``clip_and_step()`` clips and
    updates from ``p.grad`` (which this class points at the averaged bucket views once)."""

    def __init__(self, model, fwd_loss, clip_and_step, example_inputs, warmup=2, group=None):
        self.model = model
        # the captured graphs write into whatever these close over (an optimizer's state, a step counter): keep them
        # alive as long as the graphs
        self.fwd_loss, self.clip_and_step = fwd_loss, clip_and_step
        self.params_by_segment = segment_params(model)
        self.reducer = GradAllReducer(model, group=group, groups=self.params_by_segment, sinks_always=True)
        self.reducer.manual = True
        self.reducer.point_grads()
        self.static_inputs = [torch.empty_like(a).copy_(a) for a in example_inputs]
        nseg = len(SEGMENTS)

        def eager():
            model._taps = {}
            loss = fwd_loss(*self.static_inputs)
            taps, model._taps = model._taps, None
            segmented_backward(model, loss, taps, self.params_by_segment,
                               after_segment=lambda k: self.reducer.launch_bucket(k))
            self.reducer.wait_all()
            clip_and_step()
            return loss

        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):                      # warm-up on a side stream, as graph capture requires
            for _ in range(warmup):
                eager()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()

        kw = dict(capture_error_mode="thread_local")
        self.g_fwd = torch.cuda.CUDAGraph()
        model._taps = {}
        with torch.cuda.graph(self.g_fwd, **kw):
            self.static_loss = fwd_loss(*self.static_inputs)
        taps, model._taps = model._taps, None
        pool = self.g_fwd.pool()
        self.g_bwd = []
        state = {}
        views = {id(p): v for b in self.reducer.buckets for p, v in zip(b["params"], b["views"])}
        self.grad_copies = 0           # gradients a kernel could not write into their bucket view (0 for UNet)

        def seg_capture(k, outputs, grad_outputs, cut):
            g = torch.cuda.CUDAGraph()
            ps = [p for p in self.params_by_segment[k] if p.requires_grad]
            with torch.cuda.graph(g, pool=pool, **kw):
                res = torch.autograd.grad(outputs, ps + cut, grad_outputs, allow_unused=True)
                # a gradient that did not land in its bucket view (a re-layout fallback, a layout the kernel cannot
                # write) is copied there by the same graph
                for p, r in zip(ps, res):
                    v = views[id(p)]
                    if r is not None and (r.data_ptr() != v.data_ptr() or r.stride() != v.stride()):
                        v.copy_(r)
                        self.grad_copies += 1
            self.g_bwd.append(g)
            state[k] = res[:len(ps)]                       # (alias the bucket views: kept alive for clarity)
            return res[len(ps):]

        t = taps
        src = lambda *names: [t[n][0] for n in names]      # noqa: E731
        cut = lambda *names: [t[n][1] for n in names]      # noqa: E731
        g_u2, g_x2, g_x1 = seg_capture(0, [self.static_loss], None, cut("u2", "x2", "x1"))
        g_x5, g_x4, g_x3 = seg_capture(1, src("u2"), [g_u2], cut("x5", "x4", "x3"))
        (g_p3,) = seg_capture(2, src("x5", "x4"), [g_x5, g_x4], cut("p3"))
        seg_capture(3, src("x3", "p3", "x2", "x1"), [g_x3, g_p3, g_x2, g_x1], [])
        del t, taps, src, cut, g_u2, g_x2, g_x1, g_x5, g_x4, g_x3, g_p3
        self._keep = state
        self.g_opt = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.g_opt, pool=pool, **kw):
            clip_and_step()
        torch.cuda.synchronize()
        assert len(self.g_bwd) == nseg

    def describe(self):
        mb = [b["numel"] * 4 / 2 ** 20 for b in self.reducer.buckets]
        return ("on (forward graph | %d backward-segment graphs, bucket all-reduce of segment k launched on NCCL's "
                "stream while segment k+1 runs; buckets %s MiB | optimizer graph)"
                % (len(self.g_bwd), "/".join(f"{m:.1f}" for m in mb)))

    def load(self, *inputs):
        for s, a in zip(self.static_inputs, inputs):
            s.copy_(a, non_blocking=True)

    def replay(self):
        check_peer_groups()
        self.g_fwd.replay()
        for k, g in enumerate(self.g_bwd):
            g.replay()
            self.reducer.launch_bucket(k)
        self.reducer.wait_all()
        self.g_opt.replay()
        F = _functional()
        if F is not None:
            F.graph_replayed()          # the weights and running statistics moved: drop the cached operands
        return self.static_loss

    def __call__(self, *inputs):
        self.load(*inputs)
        return self.replay()

    def release(self):
        """Drop the graphs and un-register the gradient sinks (the model goes back to plain backward())."""
        self.reducer.remove()
        for p in self.reducer.params:
            p.grad = None
        self.g_fwd = self.g_opt = None
        self.g_bwd = []
        self._keep = None
