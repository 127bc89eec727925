"""Batched, overlapped host feed for video: the B200-side counterpart of the reference's
one-frame-at-a-time loop (main.py:60-71: get_image -> visualize -> render).

Frames are independent, so a batch is cut into chunks that flow through three CUDA streams:
  H2D copy of chunk i+1  ||  kernels of chunk i  ||  D2H copy of chunk i-1
from / to pinned host memory.  No collective, no host synchronisation inside the loop.
"""
from __future__ import annotations

from typing import List, Optional, Protocol, Sequence, Tuple

import numpy as np

from ._abi import check
from .engine import get_engine


class RecordSink(Protocol):
    """Where run_split_jpeg delivers its frames (renderers/mjpeg.py MjpegAviWriter is one)."""

    def write_records(self, records: memoryview, jpeg_lengths: Sequence[int]) -> None:
        """`records`: consecutive AVI '00dc' chunks (fourcc, little-endian u32 size, JPEG, zero padding to a multiple of
        4), one per frame in frame order, with the JPEG lengths.  Valid only during the call."""


class HostBatchPipeline:
    def __init__(self, device=None, chunk_frames: int = 4, depth: int = 3):
        self.eng = get_engine(device)
        t = self.eng.torch
        self.chunk = int(chunk_frames)
        self.depth = int(depth)
        with t.cuda.device(self.eng.device):
            self.s_in, self.s_run, self.s_out = (t.cuda.Stream() for _ in range(3))
            # run_split_jpeg's record copies: on s_out they would queue behind the offset copies of later chunks, which
            # wait for those chunks' kernels
            self.s_rec = t.cuda.Stream()
        self._slots = {}
        self._jpeg_slots = {}
        self._staging = [None, None]

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

    def _split_plan(self, jobs, labels, what: str):
        """[(species, frames_host, label stencil or None)] of run_split's (or run_split_jpeg's) jobs, every job and the
        labels checked."""
        from .serving import _check_labels
        t = self.eng.torch
        labels = None if labels is None else _check_labels(labels)
        plan = []
        for species, src in jobs:
            if not (isinstance(src, t.Tensor) and src.device.type == "cpu" and src.dtype == t.uint8 and src.dim() == 4
                    and src.shape[1] >= 1 and src.shape[2] >= 1 and src.shape[3] == 3 and src.is_contiguous()
                    and src.is_pinned()):
                raise ValueError(f"{what}: frames_host must be a pinned, contiguous uint8 CPU tensor [N,H,W,3]")
            h, w = src.shape[1], src.shape[2]
            plan.append((species, src, None if labels is None else self.eng.split_stencil(h, w, *labels)))
        spans = sorted((src.data_ptr(), src.data_ptr() + src.numel()) for _, src, _ in plan if src.numel())
        if any(lo < prev_hi for (_, prev_hi), (lo, _) in zip(spans, spans[1:])):
            raise ValueError(f"{what}: two jobs share host frames" +
                             ("; each job's frames are overwritten in place" if what == "run_split" else ""))
        return plan

    def run_split(self, jobs: Sequence[Tuple[object, object]], *,
                  labels: Optional[Tuple[str, str]] = ("Original", "Transformed"), draw_seam: bool = True):
        """jobs: (species, frames_host) with frames_host a pinned, contiguous uint8 CPU tensor [N,H,W,3].  Turns every
        frame, in place, into its labelled split frame (`split_compare_batch(frame, view, draw_seam=..., labels=...)`,
        the bytes of make_split_frame): per chunk H2D, visualize_batch and K9 on the device, then only the bytes that
        differ from the input come back (the label band and columns [W // 2, W), Engine.split_fetch).  `labels` is a pair
        of strings or None for none.  Jobs must not share host frames (each job's frames are uploaded and overwritten
        in place).  Every job is checked before anything is enqueued; waits once, also when a job fails mid-way, so no
        copy into the caller's frames is left in flight.  Returns (h2d_bytes, d2h_bytes) as copied."""
        t = self.eng.torch
        plan = self._split_plan(jobs, labels, "run_split")
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

    def _jpeg_bufs(self, h: int, w: int, k8):
        """`depth` rotating sets of (K8 workspace, K8 slots, packed records, device [offsets | lengths], the same pinned)
        for chunks of h x w frames, used beside _slot_bufs' buffers of the same slot index.  Like _slot_bufs they are
        kept for the pipeline's lifetime, per (h, w): at 4K in chunks of 2 about 0.5 GB of device memory per slot (K8's
        worst-case slot bound is 84 MB a frame, for the slots and again for the packed records)."""
        key = (h, w)
        if key not in self._jpeg_slots:
            t, dev, c = self.eng.torch, self.eng.device, self.chunk
            rec = 8 + ((k8.slot + 3) & ~3)
            self._jpeg_slots[key] = [
                (t.empty(k8.workspace_bytes(c), dtype=t.uint8, device=dev),
                 t.empty(c * k8.slot, dtype=t.uint8, device=dev),
                 t.empty(c * rec, dtype=t.uint8, device=dev),
                 t.empty(2 * c + 1, dtype=t.int64, device=dev),
                 t.empty(2 * c + 1, dtype=t.int64).pin_memory())
                for _ in range(self.depth)]
        return self._jpeg_slots[key]

    def _staging_for(self, k: int, nbytes: int):
        """Pinned staging buffer k (of 2) of at least nbytes; grown as needed and kept, like the slot buffers."""
        t = self.eng.torch
        if self._staging[k] is None or self._staging[k].numel() < nbytes:
            self._staging[k] = None
            self._staging[k] = t.empty(max(nbytes, 1), dtype=t.uint8).pin_memory()
        return self._staging[k]

    def run_split_jpeg(self, jobs: Sequence[Tuple[object, object]], *,
                       labels: Optional[Tuple[str, str]] = ("Original", "Transformed"), draw_seam: bool = True,
                       quality: int = 95, out: RecordSink):
        """jobs as run_split's; the frames are RGB and are not modified.  Every labelled split frame is encoded on the
        device as the bytes of `cv2.imencode(".jpg", split[..., ::-1], [IMWRITE_JPEG_QUALITY, quality])` and handed to
        `out.write_records` as an AVI '00dc' record, in frame order: per chunk H2D on s_in; visualize_batch, K9, K8 (RGB)
        and the record pack (K11) on s_run; the record offsets and JPEG lengths to pinned memory on s_out.  Chunk i is
        retired once chunks up to i + depth - 1 are enqueued: the host waits for its offsets, then copies exactly its
        record bytes into one of two pinned staging buffers on s_rec, a stream that waits for nothing but that chunk,
        and hands the previous chunk's records to `out` while this copy and the later chunks' work run.  Only
        compressed bytes cross.  Every job, the labels and the quality are checked before anything is enqueued; waits
        once at the end, also when a job fails mid-way (the chunks not yet handed to `out` then are not).  Returns
        (h2d_bytes, d2h_bytes) as copied."""
        from .jpeg import JPEG_LAUNCHES, JpegLauncher, check_quality
        t = self.eng.torch
        eng = self.eng
        plan = self._split_plan(jobs, labels, "run_split_jpeg")
        quality = check_quality(quality, "run_split_jpeg")
        if not callable(getattr(out, "write_records", None)):
            raise TypeError("run_split_jpeg: out must have write_records(records, jpeg_lengths)")
        k8s = {}
        for _, src, _ in plan:
            hw = (src.shape[1], src.shape[2])
            if hw not in k8s:
                k8s[hw] = JpegLauncher(eng.lib, *hw, quality, rgb=True)
        h2d = d2h = 0
        slot_i = 0
        pending = []                      # enqueued chunks whose records are not yet copied, oldest first
        staged = []                       # at most one (copy event, staging, bytes, lengths) not yet handed to `out`
        retired = 0

        def hand_over():
            e_out, staging, total, lengths = staged.pop()
            e_out.synchronize()
            out.write_records(memoryview(staging.numpy()[:total]), lengths)

        def retire():
            nonlocal d2h, retired
            e_meta, meta_host, packed, n, ev = pending.pop(0)
            e_meta.synchronize()          # s_out holds offset copies only, in chunk order: this waits for chunk i alone
            meta = meta_host.numpy()
            total = int(meta[n])
            lengths = [int(x) for x in meta[n + 1:2 * n + 1]]
            # buffer retired % 2 last held chunk i - 2, handed over during the previous retire
            staging = self._staging_for(retired % 2, total)
            retired += 1
            with t.cuda.stream(self.s_rec):
                self.s_rec.wait_event(e_meta)
                staging[:total].copy_(packed[:total], non_blocking=True)
                e_out = t.cuda.Event()
                e_out.record(self.s_rec)
            ev[0] = e_out
            d2h += total
            if staged:
                hand_over()
            staged.append((e_out, staging, total, lengths))

        with t.cuda.device(eng.device):
            try:
                for species, src, stencil in plan:
                    n_all, h, w = src.shape[0], src.shape[1], src.shape[2]
                    k8 = k8s[(h, w)]
                    fs, rs = h * w * 3, w * 3
                    for a in range(0, n_all, self.chunk):
                        b = min(n_all, a + self.chunk)
                        n = b - a
                        slots = self._slot_bufs((self.chunk,) + tuple(src.shape[1:]), 2)
                        d_in, (d_split, d_view), ev = slots[slot_i % self.depth]
                        ws, jslots, packed, meta, meta_host = self._jpeg_bufs(h, w, k8)[slot_i % self.depth]
                        slot_i += 1
                        if ev[0] is not None:                    # slot reused: its last D2H must be done
                            self.s_in.wait_event(ev[0])
                            self.s_run.wait_event(ev[0])
                        with t.cuda.stream(self.s_in):
                            d_in[:n].copy_(src[a:b], non_blocking=True)
                            e_in = t.cuda.Event()
                            e_in.record(self.s_in)
                        with t.cuda.stream(self.s_run):
                            self.s_run.wait_event(e_in)
                            if self.n_outputs(species) == 2:
                                species.visualize_batch(d_in[:n], out=(d_split[:n], d_view[:n]))
                            else:
                                species.visualize_batch(d_in[:n], out=d_view[:n])
                            eng.split_compose(d_in[:n], d_view[:n], d_split[:n], bool(draw_seam), stencil)
                            # meta: [0, n] the record offsets (K11), [n + 1, 2n] the JPEG lengths (K8)
                            st = eng.stream_ptr()
                            check(k8.launch(d_split.data_ptr(), n, fs, rs, ws.data_ptr(), jslots.data_ptr(), k8.slot,
                                            meta[n + 1:].data_ptr(), st), k8.name)
                            check(eng.lib.avb_mjpeg_pack_u8(jslots.data_ptr(), k8.slot, meta[n + 1:].data_ptr(), n,
                                                            packed.data_ptr(), meta.data_ptr(), st), "avb_mjpeg_pack_u8")
                            eng.launches += JPEG_LAUNCHES + 1
                            e_run = t.cuda.Event()
                            e_run.record(self.s_run)
                        with t.cuda.stream(self.s_out):
                            self.s_out.wait_event(e_run)
                            meta_host[:2 * n + 1].copy_(meta[:2 * n + 1], non_blocking=True)
                            e_meta = t.cuda.Event()
                            e_meta.record(self.s_out)
                        pending.append((e_meta, meta_host, packed, n, ev))
                        h2d += n * fs
                        d2h += (2 * n + 1) * 8
                        if len(pending) == self.depth:
                            retire()
                while pending:
                    retire()
                if staged:
                    hand_over()
            finally:
                for s in (self.s_rec, self.s_out, self.s_run, self.s_in):
                    s.synchronize()
        return h2d, d2h
