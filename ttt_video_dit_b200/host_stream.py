"""Feeding the op from HOST memory: double-buffered H2D prefetch and asynchronous D2H around any of this package's ops.

The reference keeps its activations on the device for the whole model, so it has no counterpart of this file; it exists for
callers that hold the token tensors in pinned host memory (offloaded activations, a data-loader handing over latents) and
for the end-to-end leg of bench.py.  One step moves 447 MB in and 111 MB out for the 3-second TTT-MLP workload, which at
PCIe Gen5 rates is as long as the scan itself, so the copies have to run beside the kernels rather than in front of them:

    copy-in stream :  H2D(i+1) ------------|  H2D(i+2) ------------|
    compute stream :  op(i) -------------|    op(i+1) -------------|
    copy-out stream:                      D2H(i) ---|               D2H(i+1) ---|

Every step still pays its own H2D and D2H inside the caller's timed region; only their placement changes.  Staging buffers
are allocated once per slot and reused (no allocator traffic on the side streams); ordering is by CUDA events only, the
host never blocks inside `run`.
"""
from typing import Callable, Iterable, Optional, Sequence

import torch

from . import _lib


class HostPipeline:
    """`HostPipeline(device).run(batches, fn, host_out)` calls `fn(*device_tensors)` once per batch of pinned host tensors.

    batches : iterable of tuples of pinned CPU tensors (entries may be None); all batches share shapes / dtypes
    fn      : the op, called on the compute (current) stream with the staged device tensors; returns the result tensor
    host_out: pinned CPU tensor (or a list of them, used round-robin) that receives each result
    Returns the number of steps run.  The current stream has waited for the last D2H when `run` returns, so an event
    recorded right after it brackets the whole pipeline.
    """

    def __init__(self, device, depth: int = 2):
        _lib.lib()  # the op behind `fn` is CUDA-only; fail here, loudly, when the extension is missing
        self.device = torch.device(device)
        self.depth = max(2, int(depth))
        self.s_in = torch.cuda.Stream(self.device)
        self.s_out = torch.cuda.Stream(self.device)
        self.staged = [None] * self.depth  # per-slot tuples of device tensors
        self.ev_in = [torch.cuda.Event() for _ in range(self.depth)]    # H2D into the slot finished
        self.ev_free = [torch.cuda.Event() for _ in range(self.depth)]  # the op that consumed the slot finished
        self.ev_out = torch.cuda.Event()
        self.h2d_bytes = 0
        self.d2h_bytes = 0

    def _stage(self, slot: int, host: Sequence[Optional[torch.Tensor]], first_use: bool):
        with torch.cuda.stream(self.s_in):
            if not first_use:
                self.s_in.wait_event(self.ev_free[slot])
            for d, t in zip(self.staged[slot], host):
                if t is None:
                    continue
                if not t.is_pinned():
                    raise ValueError("HostPipeline: host tensors must be pinned (torch.Tensor.pin_memory)")
                d.copy_(t, non_blocking=True)
                self.h2d_bytes += t.numel() * t.element_size()
            self.ev_in[slot].record(self.s_in)

    def run(self, batches: Iterable[Sequence[Optional[torch.Tensor]]], fn: Callable[..., torch.Tensor], host_out) -> int:
        outs = list(host_out) if isinstance(host_out, (list, tuple)) else [host_out]
        main = torch.cuda.current_stream(self.device)
        it = iter(batches)
        nxt = next(it, None)
        if nxt is None:
            return 0
        if self.staged[0] is None:
            # every slot up front: a staging block comes from the compute stream's pool and may have been freed by work still
            # running there (an earlier op's checkpoints), so it must exist before the copy stream's wait below
            self.staged = [tuple(None if t is None else torch.empty(t.shape, dtype=t.dtype, device=self.device) for t in nxt)
                           for _ in range(self.depth)]
        self.s_in.wait_stream(main)  # staging buffers / earlier users of the slots are ordered before the first copy
        self._stage(0, nxt, True)
        i = 0
        while nxt is not None:
            slot = i % self.depth
            nxt = next(it, None)
            if nxt is not None:  # prefetch batch i+1 while batch i computes
                self._stage((i + 1) % self.depth, nxt, i + 1 < self.depth)
            main.wait_event(self.ev_in[slot])
            res = fn(*self.staged[slot])
            self.ev_free[slot].record(main)
            dst = outs[i % len(outs)]
            with torch.cuda.stream(self.s_out):
                self.s_out.wait_event(self.ev_free[slot])
                dst.copy_(res.detach(), non_blocking=True)
                res.record_stream(self.s_out)
                self.d2h_bytes += dst.numel() * dst.element_size()
            i += 1
        self.ev_out.record(self.s_out)
        main.wait_event(self.ev_out)
        return i
