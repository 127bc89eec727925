"""Batched frame feed that sits beside the reference's `VideoRenderer.get_image()`
(renderers/video.py:82-96), and the labelled split-compare frame of `make_split_frame` (:198-245) for whole batches.

Video decode and encode stay on the CPU in the reference's own renderer; `BatchFeed` only gathers its frames into
pinned batches for `visualize_batch`.  The split-compare frame, corner labels included, is composed on the device
(K9, `split_compare_batch(..., labels=...)`): the labels reach the device as per-pixel byte tables built from
`draw_split_labels` itself (`tables.split_label_stencil`), so the device frame has the bytes the host drawing gives."""
from __future__ import annotations

from typing import List, NamedTuple, Optional, Tuple

import numpy as np


class BatchFeed:
    """Wraps any object with `get_image() -> Optional[np.ndarray HxWx3 uint8]` (the reference's
    VideoRenderer / WebcamRenderer / ImageRenderer all have it)."""

    def __init__(self, source, batch: int = 8, pinned: bool = True):
        self.source = source
        self.batch = int(batch)
        self.pinned = pinned
        self._buf = None

    def get_batch(self, n: Optional[int] = None):
        """Up to n frames as a uint8 array/tensor [k,H,W,3] (k <= n; None at end of stream)."""
        n = n or self.batch
        first = self.source.get_image()
        if first is None:
            return None
        assert first.ndim == 3 and first.shape[2] == 3 and first.dtype == np.uint8
        if self._buf is None or tuple(self._buf.shape[1:]) != first.shape or self._buf.shape[0] < n:
            if self.pinned:
                import torch
                self._buf = torch.empty((n,) + first.shape, dtype=torch.uint8).pin_memory()
            else:
                self._buf = np.empty((n,) + first.shape, np.uint8)
        view = self._buf.numpy() if self.pinned else self._buf
        view[0] = first
        k = 1
        while k < n:
            f = self.source.get_image()
            if f is None:
                break
            view[k] = f
            k += 1
        return self._buf[:k]


def _check_split_args(original, modified, out):
    assert original.shape == modified.shape and original.dim() == 4 and original.shape[3] == 3, "frames must be [N,H,W,3] of one shape"
    assert original.dtype == modified.dtype and original.device == modified.device
    if out is None:
        return original.new_empty(original.shape)
    assert out.shape == original.shape and out.dtype == original.dtype and out.device == original.device, \
        "out must be a tensor of the frames' shape, dtype and device"
    for name, x in (("original", original), ("modified", modified)):
        if _overlap(out, x):
            raise ValueError(f"split_compare_batch: out overlaps {name}")
    return out


def _overlap(a, b) -> bool:
    """Whether the byte extents of two tensors intersect (conservative: extents, not individual elements)."""
    if a.numel() == 0 or b.numel() == 0 or a.untyped_storage().data_ptr() != b.untyped_storage().data_ptr():
        return False

    def extent(x):
        lo = x.data_ptr()
        return lo, lo + sum((s - 1) * st for s, st in zip(x.shape, x.stride())) * x.element_size() + x.element_size()
    (a0, a1), (b0, b1) = extent(a), extent(b)
    return a0 < b1 and b0 < a1


def split_compare_batch(original, modified, out=None, *, draw_seam: bool = True,
                        labels: Optional[Tuple[str, str]] = None):
    """`make_split_frame` (reference renderers/video.py:198-245) for a whole batch: left half of `original`, right half
    of `modified`, optional 1-px white seam at W // 2, and with `labels=(left, right)` the two corner labels, the bytes
    `draw_split_labels(frame, left, right)` draws.  Tensors are uint8 [N,H,W,3] of one shape on one device; `out` (same
    shape, any frame / row strides, packed pixels) must not overlap either input.

    CUDA tensors go through one kernel (K9, `avb_split_compose_u8`) on the current stream, labelled or not, and the frames
    never visit the host; the label tables are built once per (H, W, labels) and device.  CPU tensors take strided slice
    copies and accept no labels: draw them with `draw_split_labels` on the host frames.  (The reference's INTER_AREA
    resize of a mismatching `modified` is not needed: every species returns frames of the input's shape.)"""
    out = _check_split_args(original, modified, out)
    if original.is_cuda:
        from ..engine import get_engine
        eng = get_engine(original.device)
        stencil = None if labels is None else eng.split_stencil(original.shape[1], original.shape[2], *labels)
        eng.split_compose(original, modified, out, bool(draw_seam), stencil)
        return out
    if labels is not None:
        raise ValueError("split_compare_batch: labels need CUDA tensors; on host frames call draw_split_labels")
    mid = original.shape[2] // 2
    out[:, :, :mid].copy_(original[:, :, :mid])
    out[:, :, mid:].copy_(modified[:, :, mid:])
    if draw_seam:
        out[:, :, mid:mid + 1] = 255
    return out


class LabelBox(NamedTuple):
    """One corner label of the split frame: its text, putText origin, scale and thickness, and the backing rectangle
    (x0, y0, x1, y1), inclusive, already clamped to the frame."""
    text: str
    org: Tuple[int, int]
    scale: float
    thickness: int
    rect: Tuple[int, int, int, int]


LABEL_FONT_COLOURS = ((0, 0, 0), (255, 255, 255))           # outline, then fill (renderers/video.py:160-196)


def split_label_geometry(H: int, W: int, left_label: str = "Original", right_label: str = "Transformed") -> List[LabelBox]:
    """Where `draw_split_labels` puts the two labels of an H x W frame (`_draw_label`, renderers/video.py:160-196, called
    at :241-244).  Depends on H, W and the texts only."""
    import cv2
    font = cv2.FONT_HERSHEY_SIMPLEX

    def label(text, org):
        scale, thickness, pad = max(0.5, min(1.2, H / 900.0)), 2, 8
        (tw, th), baseline = cv2.getTextSize(text, font, scale, thickness)
        x, y = org
        if x + tw + pad > W:                                   # keep inside the frame
            x = W - tw - pad
        if y - th - baseline - pad < 0:
            y = th + baseline + pad
        x0, y0 = max(x - pad, 0), max(y - th - baseline - pad, 0)
        x1, y1 = min(x + tw + pad, W - 1), min(y + baseline + pad, H - 1)
        return LabelBox(text, (x, y), scale, thickness, (x0, y0, x1, y1))
    (tw, _), _ = cv2.getTextSize(right_label, font, max(0.45, min(1.2, H / 900.0)), 1)      # :242: its own scale / thickness
    return [label(left_label, (10, 24)), label(right_label, (max(W - tw - 10, 10), 24))]


def draw_label_boxes(frame: np.ndarray, boxes: List[LabelBox]) -> np.ndarray:
    """Draw labels placed by `split_label_geometry` onto `frame` (any number of rows: drawing is clipped to it), in place:
    darken the rectangle to 40 %, then the text outlined in black and filled in white, anti-aliased."""
    import cv2
    font = cv2.FONT_HERSHEY_SIMPLEX
    outline, fill = LABEL_FONT_COLOURS
    for b in boxes:
        x0, y0, x1, y1 = b.rect
        overlay = frame.copy()
        cv2.rectangle(overlay, (x0, y0), (x1, y1), (0, 0, 0), thickness=-1)
        cv2.addWeighted(overlay, 0.6, frame, 0.4, 0, frame)
        cv2.putText(frame, b.text, b.org, font, b.scale, outline, b.thickness + 2, cv2.LINE_AA)
        cv2.putText(frame, b.text, b.org, font, b.scale, fill, b.thickness, cv2.LINE_AA)
    return frame


def draw_split_labels(frame: np.ndarray, left_label: str = "Original", right_label: str = "Transformed") -> np.ndarray:
    """The label step of `make_split_frame` (renderers/video.py:160-196 `_draw_label`, :241-244) on one host frame, in place."""
    H, W = frame.shape[:2]
    return draw_label_boxes(frame, split_label_geometry(H, W, left_label, right_label))
