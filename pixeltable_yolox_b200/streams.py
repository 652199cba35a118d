"""Side streams for the independent branches of the training step.

At 8 images per GPU every kernel of the step is a fraction of a wave; the step is a chain of ~1 100 launches whose length,
not whose work, sets the time. The network has branches that do not depend on each other -- the two 1x1 convs at the head of
a CspLayer (yolox/models/network_blocks.py:176-177), the three levels of YoloxHead and its cls / reg towers
(yolox/models/yolo_head.py:140-160) -- and a `Branch` runs one of them on a side stream: fork = the side stream waits for an
event recorded on the current stream, join = the current stream waits for the side stream. Autograd replays every backward
node on the stream its forward ran on and inserts the matching waits, so the backward of a branch overlaps as well; a CUDA
graph capture records forks and joins as graph branches.

Memory: tensors cross streams only over a fork or a join, and every tensor a branch produces is kept alive by autograd until
its backward, i.e. long after its consumers on the other stream were enqueued; every later fork orders the side stream after all
earlier work of the forking stream, so the caching allocator's per-stream reuse stays ordered (no record_stream needed, which
a graph capture would not allow).
"""
from __future__ import annotations

import torch

_streams = {}


def side_stream(dev: torch.device, idx: int) -> "torch.cuda.Stream":
    key = (dev.index if dev.index is not None else torch.cuda.current_device(), idx)
    s = _streams.get(key)
    if s is None:
        s = _streams[key] = torch.cuda.Stream(dev)
    return s


_ready = {}


def mark_ready(x: torch.Tensor) -> torch.Tensor:
    """Record "x is complete" on the current stream; a Branch created on x later forks from this point instead of from the
    point of its creation (YoloPafpn: the stride-8 head level only needs pan_out2, not the bottom-up half of the neck)."""
    if enabled(x):
        import weakref

        _ready[id(x)] = (weakref.ref(x), torch.cuda.current_stream(x.device).record_event())
    return x


def enabled(x: torch.Tensor) -> bool:
    return x.is_cuda


class Branch:
    """`br = Branch(x, 3); with br: y = f(x)` runs f on side stream 3 of x's device, forked from the current stream now;
    `br.join()` makes the (then) current stream wait for it. With `enabled(x)` false everything runs in line."""

    def __init__(self, x: torch.Tensor, idx: int):
        self.on = enabled(x)
        if self.on:
            self.dev = x.device
            self.side = side_stream(self.dev, idx)
            # fork point: the event `mark_ready` attached to x when it was produced (the branch then overlaps whatever the
            # producing stream enqueued after x), else "now"
            ev = _ready.pop(id(x), None)
            self.side.wait_event(ev[1] if ev is not None and ev[0]() is x else torch.cuda.current_stream(self.dev).record_event())
            self.ctx = None

    def __enter__(self):
        if self.on:
            self.ctx = torch.cuda.stream(self.side)
            self.ctx.__enter__()
        return self

    def __exit__(self, *exc):
        if self.on:
            self.ctx.__exit__(*exc)
        return False

    def join(self) -> None:
        if self.on:
            torch.cuda.current_stream(self.dev).wait_event(self.side.record_event())
