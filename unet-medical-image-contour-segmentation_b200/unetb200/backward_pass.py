"""The work a backward pass of the library's Functions leaves outside autograd, owned by one record per autograd
graph task (`_Pass`), made the first time the pass needs one: split reductions deferred to the end of the pass
(`defer_reduce`), the operands and the join of weight gradients on the side stream (`on_side_stream`), and gradient
hand-offs from the kernel that writes a gradient to its consumer (`leave` / `take`).

One engine callback at the end of the pass reduces the queued jobs by one launch, joins the side stream, releases the
operands and discards the hand-offs nobody took.  A pass that raises never runs its callbacks: a record of a graph task
other than the running one belongs to such a pass, and is dropped before a new record is made or a forward pass starts.
"""
from __future__ import annotations

import contextlib

import torch

from . import _lib, ops

# ------------------------------------------------------------------------------------------------
# deferred split reductions of the weight gradients: one multi-tensor launch for several layers
# ------------------------------------------------------------------------------------------------
# A wgrad kernel writes `splits` partial results; reducing them layer by layer costs 22 small launches per step.
# Two ways to batch them, both chosen per layer by functional (gconv_wgrad's `defer`):
# * "call": the reductions queued while one Function's backward runs (functional.DoubleConvFn: both of its convs;
#   UpCatConvTFn: its ConvTranspose) are made by ONE launch when that backward returns (`reductions_at_return`).
#   Autograd only sees the gradients after that, so everything that reads them during the pass -- AccumulateGrad and
#   hooks on its node (where stock DistributedDataParallel and FSDP attach), the engine summing the two contributions
#   of a parameter used twice -- reads finished values.
# * "pass": when a data-parallel sink owns the gradient (functional._sink_owns: the reducer drives the pass through
#   torch.autograd.grad and is its only reader), the reduction is queued in the pass's record and all queued layers
#   are reduced by ONE launch at the end of the pass -- for a segmented backward (ddp.segmented_backward) that is the
#   end of each torch.autograd.grad call, i.e. before the segment's bucket is all-reduced.
# NOTE a job keeps the partials alive but only the ADDRESS of the gradient: AccumulateGrad adopts a gradient tensor
# without copying only while nobody else references it (use_count check) -- a reference held here would make it clone
# the not-yet-reduced buffer.  Switch: ops.DEFER_REDUCE.

# ------------------------------------------------------------------------------------------------
# side stream for weight gradients
# ------------------------------------------------------------------------------------------------
# A weight gradient is needed only by the optimizer, while the BatchNorm backward of the previous layer (HBM bound,
# few registers, no shared memory) needs the data gradient and is what autograd runs next.  Issuing the wgrad GEMM
# on a second stream -- ordered after the dgrad of the same layer -- lets the memory-bound kernels of the next
# layer run on the SM resources the tensor kernel leaves idle.  The streams are joined at the end of the backward
# pass (so callers such as the reference train.py need no change), and the operands are kept alive until then.
# Switches: ops._SIDE_ON, ops._WGRAD_SIDE.
_SIDE = {}            # device index -> torch.cuda.Stream


def graph_task():
    """Id of the autograd graph task running on this thread (< 0 outside a backward pass)."""
    return torch._C._current_graph_task_id()


class _Pass:
    """Everything one backward pass (autograd graph task) owns outside autograd until it ends."""
    __slots__ = ("task", "jobs", "keep", "join", "handoffs")

    def __init__(self, task):
        self.task = task
        self.jobs = []          # "pass" jobs: (partials, dst address, st, sc, sq, sn, splits, ntaps, Cin, N, Cq)
        self.keep = []          # tensors the side stream still reads
        self.join = False       # the side stream is to be joined at the end of the pass
        self.handoffs = {}      # (kind, data_ptr(g)) -> (value, shape of g, token)


_PASS = [None]          # the record of the last backward pass that needed one (None once it has ended)
_CALL_JOBS = [None]     # the "call" jobs of the Function backward running now (None: outside reductions_at_return)


def _drop():
    """Forget the record of a backward pass that raised before its end-of-pass callback ran: order the current stream
    after the side stream (its kernels may still write into tensors of the failed pass), then drop the queued
    reductions -- their destinations may have been freed and handed out again --, the operands and the hand-offs."""
    side_stream_sync()
    _PASS[0] = None


def _record():
    """The record of the running backward pass, made (with its end-of-pass callback) on first use; None outside a
    backward pass.  A record of another graph task belongs to a pass that raised: it is dropped first."""
    task = graph_task()
    rec = _PASS[0]
    if rec is not None and rec.task != task:
        _drop()
        rec = None
    if rec is None and task >= 0:
        rec = _PASS[0] = _Pass(task)
        torch.autograd.Variable._execution_engine.queue_callback(lambda: _end_of_pass(rec))
    return rec


def _end_of_pass(rec):
    """The engine callback of `rec`'s pass: reduce its queued jobs by one launch on the current stream, join the side
    stream, then let go of the operands and of the hand-offs nobody took."""
    if _PASS[0] is not rec:
        return                      # dropped for a pass of another graph task
    _PASS[0] = None
    _reduce_multi(rec.jobs)
    if rec.join:
        side_stream_sync()
    rec.keep.clear()
    rec.handoffs.clear()


def begin_forward():
    """Entry of a drop-in forward pass.  Outside any backward pass, a record still held belongs to a pass that raised
    (train.py's OOM retry takes this route): drop it before it can reach the next pass.  Inside one (re-computation
    under use_checkpointing) nothing changes."""
    if _PASS[0] is not None and graph_task() < 0:
        _drop()


# ------------------------------------------------------------------------------------------------
# split reductions
# ------------------------------------------------------------------------------------------------
def _reduce_multi(jobs):
    if not jobs:
        return
    arr = (_lib.ReduceJob * len(jobs))()
    nbytes = 0.0
    for j, (partials, dst, st, sc, sq, sn, splits, ntaps, Cin, N, Cq) in enumerate(jobs):
        arr[j].partials, arr[j].dst = partials.data_ptr(), dst
        arr[j].st, arr[j].sc, arr[j].sq, arr[j].sn = st, sc, sq, sn
        arr[j].splits, arr[j].ntaps, arr[j].Cin, arr[j].N, arr[j].Cq, arr[j].accumulate = splits, ntaps, Cin, N, Cq, 0
        nbytes += 4.0 * ntaps * Cin * N * (splits + 1)
    n = len(jobs)
    ops._run("wgrad_reduce", ops.lib().unetb200_wgrad_reduce_multi, arr, n, ops._stream(), nbytes=nbytes,
             kernels=(n + 31) // 32)


def defer_reduce(job, when):
    """Take the split reduction `job` of a weight gradient for one launch with others: when="call" at the end of the
    enclosing reductions_at_return block, when="pass" at the end of the backward pass (at once outside one).  False
    when it is not taken (UNETB200_DEFER_REDUCE=0, or "call" outside such a block): the caller reduces it now."""
    if not ops.DEFER_REDUCE:
        return False
    if when == "call":
        if _CALL_JOBS[0] is None:
            return False
        _CALL_JOBS[0].append(job)
        return True
    rec = _record()
    if rec is None:
        _reduce_multi([job])                         # not inside a backward pass: nothing to wait for
    else:
        rec.jobs.append(job)
    return True


@contextlib.contextmanager
def reductions_at_return():
    """The "call" reductions queued inside the block are made by one launch when it ends without an exception."""
    prev, _CALL_JOBS[0] = _CALL_JOBS[0], []
    try:
        yield
        jobs = _CALL_JOBS[0]
    finally:
        _CALL_JOBS[0] = prev
    _reduce_multi(jobs)


# ------------------------------------------------------------------------------------------------
# side stream
# ------------------------------------------------------------------------------------------------
def _wait_side(s):
    """current stream waits for side stream `s` -- unless a CUDA-graph capture is in progress that `s` is not part
    of (a captured stream may not wait on work outside its capture; there is then nothing pending on `s` either)."""
    cur = torch.cuda.current_stream(s.device)
    if torch.cuda.is_current_stream_capturing():
        with torch.cuda.stream(s):
            if not torch.cuda.is_current_stream_capturing():
                return
    cur.wait_stream(s)


def side_stream_sync():
    """Order the current stream after the side stream (for code that reads weight gradients DURING backward); no-op
    while no side stream exists."""
    for s in _SIDE.values():
        _wait_side(s)


def wgrad_on_side_stream():
    """True when weight gradients are to be computed by on_side_stream."""
    return ops._SIDE_ON and ops._WGRAD_SIDE and ops._PROFILE is None


def on_side_stream(fn, *keep):
    """Run fn() on the side stream, ordered after everything enqueued so far on the current stream.  The current
    stream is ordered after the side stream at the end of the backward pass (at once outside one), and `keep` -- the
    tensors fn's kernels read -- stays alive until then."""
    rec = _record()
    dev = torch.cuda.current_device()
    side = _SIDE.get(dev)
    if side is None:
        side = _SIDE[dev] = torch.cuda.Stream(device=dev)
    ev = torch.cuda.Event()
    ev.record(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        side.wait_event(ev)
        out = fn()
    if rec is None:
        side_stream_sync()
    else:
        rec.keep.extend(keep)
        rec.join = True
    return out


# ------------------------------------------------------------------------------------------------
# gradient hand-offs
# ------------------------------------------------------------------------------------------------
def leave(kind, g, value, token=None):
    """Hand `value`, made by the kernel that wrote the gradient `g`, to the consumer of `g` in this backward pass (none
    outside a backward pass).  `token`: the consumer's per-call object, so that an entry can never be mistaken for
    another call's (addresses repeat once the allocator recycles a block)."""
    rec = _record()
    if rec is not None:
        rec.handoffs[(kind, g.data_ptr())] = (value, tuple(g.shape), token)


def take(kind, g, token=None):
    """The value left for `g` in this backward pass with the same shape and token, else None (the entry goes either
    way)."""
    rec = _PASS[0]
    if rec is None or rec.task != graph_task():
        return None
    ent = rec.handoffs.pop((kind, g.data_ptr()), None)
    if ent is None or ent[1] != tuple(g.shape) or ent[2] is not token:
        return None
    return ent[0]
