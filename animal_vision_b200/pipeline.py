"""Batched, overlapped host feed for video: the B200-side counterpart of the reference's
one-frame-at-a-time loop (main.py:60-71: get_image -> visualize -> render).

Frames are independent, so a batch is cut into chunks that flow through three CUDA streams:
  H2D copy of chunk i+1  ||  kernels of chunk i  ||  D2H copy of chunk i-1
from / to pinned host memory.  No collective, no host synchronisation inside the loop.
"""
from __future__ import annotations

from typing import List, Optional, Sequence, Tuple

import numpy as np

from .engine import get_engine


class HostBatchPipeline:
    def __init__(self, device=None, chunk_frames: int = 4, depth: int = 3):
        self.eng = get_engine(device)
        t = self.eng.torch
        self.chunk = int(chunk_frames)
        self.depth = int(depth)
        with t.cuda.device(self.eng.device):
            self.s_in, self.s_run, self.s_out = (t.cuda.Stream() for _ in range(3))
        self._slots = {}

    def _slot_bufs(self, shape, n_out):
        """`depth` rotating device buffers: one input + n_out outputs of `shape` ([chunk,H,W,3])."""
        key = (tuple(shape), n_out)
        if key not in self._slots:
            t = self.eng.torch
            self._slots[key] = [
                (t.empty(shape, dtype=t.uint8, device=self.eng.device),
                 [t.empty(shape, dtype=t.uint8, device=self.eng.device) for _ in range(n_out)],
                 [None, None])       # [event: outputs copied out (slot free), unused]
                for _ in range(self.depth)]
        return self._slots[key]

    @staticmethod
    def n_outputs(species) -> int:
        return int(getattr(species, "N_OUTPUTS", 1))         # class attribute: Cat (and its subclasses) produce two frames

    def pinned_like(self, frames, n_out: int):
        t = self.eng.torch
        return [t.empty(tuple(frames.shape), dtype=t.uint8).pin_memory() for _ in range(n_out)]

    def run(self, jobs: Sequence[Tuple[object, object, List[object]]]):
        """jobs: (species, frames_host, outs_host) with frames_host / outs_host pinned uint8
        tensors [N,H,W,3] (outs_host: one tensor per species output, see n_outputs).
        Enqueues everything, then waits once.  Returns (h2d_bytes, d2h_bytes)."""
        t = self.eng.torch
        h2d = d2h = 0
        slot_i = 0
        with t.cuda.device(self.eng.device):
            for species, src, outs in jobs:
                n = src.shape[0]
                n_out = len(outs)
                for a in range(0, n, self.chunk):
                    b = min(n, a + self.chunk)
                    shape = (self.chunk,) + tuple(src.shape[1:])
                    slots = self._slot_bufs(shape, n_out)
                    d_in, d_outs, ev = slots[slot_i % self.depth]
                    slot_i += 1
                    if ev[0] is not None:                    # slot reused: its last D2H must be done
                        self.s_in.wait_event(ev[0])
                        self.s_run.wait_event(ev[0])
                    with t.cuda.stream(self.s_in):
                        d_in[: b - a].copy_(src[a:b], non_blocking=True)
                        e_in = t.cuda.Event()
                        e_in.record(self.s_in)
                    with t.cuda.stream(self.s_run):
                        self.s_run.wait_event(e_in)
                        if n_out == 2:
                            species.visualize_batch(d_in[: b - a], out=(d_outs[0][: b - a], d_outs[1][: b - a]))
                        else:
                            species.visualize_batch(d_in[: b - a], out=d_outs[0][: b - a])
                        e_run = t.cuda.Event()
                        e_run.record(self.s_run)
                    with t.cuda.stream(self.s_out):
                        self.s_out.wait_event(e_run)
                        for d, o in zip(d_outs, outs):
                            o[a:b].copy_(d[: b - a], non_blocking=True)
                        e_out = t.cuda.Event()
                        e_out.record(self.s_out)
                    ev[0] = e_out
                    h2d += (b - a) * int(np.prod(src.shape[1:]))
                    d2h += n_out * (b - a) * int(np.prod(src.shape[1:]))
            self.s_out.synchronize()
            self.s_run.synchronize()
        return h2d, d2h

    def run_split(self, jobs: Sequence[Tuple[object, object]], *,
                  labels: Optional[Tuple[str, str]] = ("Original", "Transformed"), draw_seam: bool = True):
        """jobs: (species, frames_host) with frames_host a pinned, contiguous uint8 CPU tensor [N,H,W,3].  Turns every
        frame, in place, into its labelled split frame (`split_compare_batch(frame, view, draw_seam=..., labels=...)`,
        the bytes of make_split_frame): per chunk H2D, visualize_batch and K9 on the device, then only the bytes that
        differ from the input come back (the label band and columns [W // 2, W), Engine.split_fetch).  `labels` is a pair
        of strings or None for none.  Jobs must not share host frames (each job's frames are uploaded and overwritten
        in place).  Every job is checked before anything is enqueued; waits once, also when a job fails mid-way, so no
        copy into the caller's frames is left in flight.  Returns (h2d_bytes, d2h_bytes) as copied."""
        from .serving import _check_labels
        t = self.eng.torch
        labels = None if labels is None else _check_labels(labels)
        plan = []
        for species, src in jobs:
            if not (isinstance(src, t.Tensor) and src.device.type == "cpu" and src.dtype == t.uint8 and src.dim() == 4
                    and src.shape[1] >= 1 and src.shape[2] >= 1 and src.shape[3] == 3 and src.is_contiguous()
                    and src.is_pinned()):
                raise ValueError("run_split: frames_host must be a pinned, contiguous uint8 CPU tensor [N,H,W,3]")
            h, w = src.shape[1], src.shape[2]
            plan.append((species, src, None if labels is None else self.eng.split_stencil(h, w, *labels)))
        spans = sorted((src.data_ptr(), src.data_ptr() + src.numel()) for _, src, _ in plan if src.numel())
        if any(lo < prev_hi for (_, prev_hi), (lo, _) in zip(spans, spans[1:])):
            raise ValueError("run_split: two jobs share host frames; each job's frames are overwritten in place")
        h2d = d2h = 0
        slot_i = 0
        with t.cuda.device(self.eng.device):
            try:
                for species, src, stencil in plan:
                    n = src.shape[0]
                    band = 0 if stencil is None else stencil[0]
                    for a in range(0, n, self.chunk):
                        b = min(n, a + self.chunk)
                        # two buffers per slot for every species: [0] the split frame (and, first, the scratch
                        # baseline of a two-output species, which the compose overwrites), [1] the view
                        slots = self._slot_bufs((self.chunk,) + tuple(src.shape[1:]), 2)
                        d_in, (d_split, d_view), ev = slots[slot_i % self.depth]
                        slot_i += 1
                        if ev[0] is not None:                    # slot reused: its last D2H must be done
                            self.s_in.wait_event(ev[0])
                            self.s_run.wait_event(ev[0])
                        with t.cuda.stream(self.s_in):
                            d_in[: b - a].copy_(src[a:b], non_blocking=True)
                            e_in = t.cuda.Event()
                            e_in.record(self.s_in)
                        with t.cuda.stream(self.s_run):
                            self.s_run.wait_event(e_in)
                            if self.n_outputs(species) == 2:
                                species.visualize_batch(d_in[: b - a], out=(d_split[: b - a], d_view[: b - a]))
                            else:
                                species.visualize_batch(d_in[: b - a], out=d_view[: b - a])
                            self.eng.split_compose(d_in[: b - a], d_view[: b - a], d_split[: b - a], bool(draw_seam),
                                                   stencil)
                            e_run = t.cuda.Event()
                            e_run.record(self.s_run)
                        # The fetch writes src[a:b], the frames the H2D above reads: it waits for e_run, recorded
                        # after the compose on s_run, which waited for e_in, recorded after that H2D.  No other
                        # chunk reads these frames (jobs do not overlap, checked above).
                        with t.cuda.stream(self.s_out):
                            self.s_out.wait_event(e_run)
                            d2h += self.eng.split_fetch(d_split[: b - a], src[a:b], band)
                            e_out = t.cuda.Event()
                            e_out.record(self.s_out)
                        ev[0] = e_out
                        h2d += (b - a) * int(np.prod(src.shape[1:]))
            finally:
                for s in (self.s_out, self.s_run, self.s_in):
                    s.synchronize()
        return h2d, d2h
