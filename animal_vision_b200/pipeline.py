"""Batched, overlapped host feed for video: the B200-side counterpart of the reference's
one-frame-at-a-time loop (main.py:60-71: get_image -> visualize -> render).

Frames are independent, so a batch is cut into chunks that flow through three CUDA streams:
  H2D copy of chunk i+1  ||  kernels of chunk i  ||  D2H copy of chunk i-1
from / to pinned host memory.  No collective, no host synchronisation inside the loop.
"""
from __future__ import annotations

from contextlib import contextmanager
from typing import List, Optional, Protocol, Sequence, Tuple

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

    @contextmanager
    def _draining(self):
        """Runs the enclosed code on the pipeline's device, then waits for all four streams, also when that code raises,
        so no copy from or into the caller's host memory outlives the call."""
        with self.eng.torch.cuda.device(self.eng.device):
            try:
                yield
            finally:
                for s in (self.s_rec, self.s_out, self.s_run, self.s_in):
                    s.synchronize()

    def _chunks(self, jobs):
        """The chunk loop of every entry point.  jobs: (job, n_buf) with job[1] its frames_host [N,H,W,3].  Per chunk
        of `chunk` frames, in job and frame order: takes the next of the `depth` slots of (chunk shape, n_buf) buffers
        (slot numbers start at 0 on each call and run on across jobs); if the slot was used before, makes s_in and s_run
        wait for its release event; uploads frames_host[a:b] on s_in and makes s_run wait for that upload (e_in).  Then
        yields (job, a, b, the device input, the n_buf device buffers, the slot's event cell, the slot number), each
        buffer cut to b - a frames.  The caller enqueues the chunk's work after e_in and sets the cell [0] to the event
        that frees the slot.  A chunk is prepared only when the caller asks for it, so it sees a release event set after
        the previous yield (run_split_jpeg sets it only when it retires a chunk)."""
        t = self.eng.torch
        slot_i = 0
        for job, n_buf in jobs:
            src = job[1]
            n = src.shape[0]
            for a in range(0, n, self.chunk):
                b = min(n, a + self.chunk)
                k = slot_i % self.depth
                d_in, d_outs, ev = self._slot_bufs((self.chunk,) + tuple(src.shape[1:]), n_buf)[k]
                slot_i += 1
                if ev[0] is not None:                    # slot reused: its last copy out must be done
                    self.s_in.wait_event(ev[0])
                    self.s_run.wait_event(ev[0])
                with t.cuda.stream(self.s_in):
                    d_in[: b - a].copy_(src[a:b], non_blocking=True)
                    e_in = self.s_in.record_event()
                self.s_run.wait_event(e_in)
                yield job, a, b, d_in[: b - a], [d[: b - a] for d in d_outs], ev, k

    def _visualize(self, species, d_in, bufs):
        """visualize_batch of d_in into slot buffers: (bufs[0], bufs[1]) for a two-output species (n_outputs), else its
        view into bufs[-1]."""
        species.visualize_batch(d_in, out=(bufs[0], bufs[1]) if self.n_outputs(species) == 2 else bufs[-1])

    def run(self, jobs: Sequence[Tuple[object, object, List[object]]]):
        """jobs: (species, frames_host, outs_host) with frames_host / outs_host pinned uint8
        tensors [N,H,W,3] (outs_host: one tensor per species output, see n_outputs).
        Enqueues everything, then waits once, also when a job fails mid-way, so no copy from or into the caller's
        tensors is left in flight.  Returns (h2d_bytes, d2h_bytes)."""
        t = self.eng.torch
        h2d = d2h = 0
        with self._draining():
            for (species, _, outs), a, b, d_in, bufs, ev, _ in self._chunks((job, len(job[2])) for job in jobs):
                with t.cuda.stream(self.s_run):
                    self._visualize(species, d_in, bufs)
                    e_run = self.s_run.record_event()
                with t.cuda.stream(self.s_out):
                    self.s_out.wait_event(e_run)
                    for d, o in zip(bufs, outs):
                        o[a:b].copy_(d, non_blocking=True)
                    ev[0] = self.s_out.record_event()
                h2d += d_in.numel()
                d2h += len(outs) * d_in.numel()
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
        with self._draining():
            # two buffers per slot for every species: [0] the split frame (and, first, the scratch baseline of a
            # two-output species, which the compose overwrites), [1] the view
            for (species, src, stencil), a, b, d_in, (d_split, d_view), ev, _ in self._chunks((j, 2) for j in plan):
                with t.cuda.stream(self.s_run):
                    self._visualize(species, d_in, (d_split, d_view))
                    self.eng.split_compose(d_in, d_view, d_split, bool(draw_seam), stencil)
                    e_run = self.s_run.record_event()
                # The fetch writes src[a:b], the frames the chunk's H2D reads: it waits for e_run, recorded after the
                # compose on s_run, which waited for e_in, recorded after that H2D (_chunks).  No other chunk reads
                # these frames (jobs do not overlap, checked above).
                with t.cuda.stream(self.s_out):
                    self.s_out.wait_event(e_run)
                    d2h += self.eng.split_fetch(d_split, src[a:b], 0 if stencil is None else stencil[0])
                    ev[0] = self.s_out.record_event()
                h2d += d_in.numel()
        return h2d, d2h

    def _jpeg_bufs(self, h: int, w: int, k8):
        """`depth` rotating sets of (K8 workspace, K8 slots, packed records, device [offsets | lengths], the same pinned)
        for chunks of h x w frames, used beside _slot_bufs' buffers of the same slot index.  Like _slot_bufs they are
        kept for the pipeline's lifetime, per (h, w) and K8 mode (the optimized mode's workspace is larger): at 4K in
        chunks of 2 about 0.5 GB of device memory per slot (K8's worst-case slot bound is 84 MB a frame, for the slots
        and again for the packed records)."""
        key = (h, w, k8.optimize)
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
                       quality: int = 95, optimize: bool = False, out: RecordSink):
        """jobs as run_split's; the frames are RGB and are not modified.  Every labelled split frame is encoded on the
        device as the bytes of `cv2.imencode(".jpg", split[..., ::-1], [IMWRITE_JPEG_QUALITY, quality])` (with
        IMWRITE_JPEG_OPTIMIZE as well if `optimize`: each frame's own Huffman tables, in its own record) and handed to
        `out.write_records` as an AVI '00dc' record, in frame order: per chunk H2D on s_in; visualize_batch, K9, K8 (RGB)
        and the record pack (K11) on s_run; the record offsets and JPEG lengths to pinned memory on s_out.  Chunk i is
        retired once chunks up to i + depth - 1 are enqueued: the host waits for its offsets, then copies exactly its
        record bytes into one of two pinned staging buffers on s_rec, a stream that waits for nothing but that chunk,
        and hands the previous chunk's records to `out` while this copy and the later chunks' work run.  Only
        compressed bytes cross.  Every job, the labels and the quality are checked before anything is enqueued; waits
        once at the end, also when a job fails mid-way (the chunks not yet handed to `out` then are not).  Returns
        (h2d_bytes, d2h_bytes) as copied."""
        from .jpeg import JpegLauncher, check_quality
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
                k8s[hw] = JpegLauncher(eng.lib, *hw, quality, rgb=True, optimize=bool(optimize))
        h2d = d2h = 0
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

        with self._draining():
            for (species, src, stencil), a, b, d_in, (d_split, d_view), ev, k in self._chunks((j, 2) for j in plan):
                n, h, w = b - a, src.shape[1], src.shape[2]
                k8 = k8s[(h, w)]
                ws, jslots, packed, meta, meta_host = self._jpeg_bufs(h, w, k8)[k]
                with t.cuda.stream(self.s_run):
                    self._visualize(species, d_in, (d_split, d_view))
                    eng.split_compose(d_in, d_view, d_split, bool(draw_seam), stencil)
                    # meta: [0, n] the record offsets (K11), [n + 1, 2n] the JPEG lengths (K8)
                    st = eng.stream_ptr()
                    check(k8.launch(d_split.data_ptr(), n, h * w * 3, w * 3, ws.data_ptr(), jslots.data_ptr(), k8.slot,
                                    meta[n + 1:].data_ptr(), st), k8.name)
                    check(eng.lib.avb_mjpeg_pack_u8(jslots.data_ptr(), k8.slot, meta[n + 1:].data_ptr(), n,
                                                    packed.data_ptr(), meta.data_ptr(), st), "avb_mjpeg_pack_u8")
                    eng.launches += k8.launches + 1
                    e_run = self.s_run.record_event()
                with t.cuda.stream(self.s_out):
                    self.s_out.wait_event(e_run)
                    meta_host[:2 * n + 1].copy_(meta[:2 * n + 1], non_blocking=True)
                    e_meta = self.s_out.record_event()
                pending.append((e_meta, meta_host, packed, n, ev))
                h2d += d_in.numel()
                d2h += (2 * n + 1) * 8
                if len(pending) == self.depth:
                    retire()
            while pending:
                retire()
            if staged:
                hand_over()
        return h2d, d2h
