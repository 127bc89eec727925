"""Device PNG encode (K10, include/avb200.h avb_png_encode_u8): the bytes of `cv2.imencode(".png", frame)` with
OpenCV's defaults for a batch of frames, computed on the GPU.  Only the compressed bytes cross to the host."""
from __future__ import annotations

from typing import List

import numpy as np

from . import tables
from ._abi import AvbError
from ._slots import encode_slots
from .engine import _fptr, get_engine


def encode_png(frames) -> List[bytes]:
    """frames: CUDA uint8 tensor [N,H,W,3] in the channel order cv2.imencode expects (BGR), packed pixels, any row
    and frame strides.  Runs on the current stream; returns one PNG file per frame."""
    import torch
    if not (isinstance(frames, torch.Tensor) and frames.is_cuda):
        raise AvbError("encode_png: expected a CUDA uint8 tensor [N,H,W,3]")
    eng = get_engine(frames.device)
    n, h, w, fs, rs = eng.check_frames(frames)
    if n == 0:
        return []
    if not (1 <= h <= 65535 and 1 <= w <= 65535):
        raise AvbError(f"encode_png: frame size {h}x{w} outside [1, 65535]^2")
    header = np.frombuffer(tables.png_header(h, w), np.uint8)
    with torch.cuda.device(eng.device):
        lib = eng.lib
        return encode_slots(
            eng, "png", n, int(lib.avb_png_bound_bytes(h, w)), int(lib.avb_png_workspace_bytes(n, h, w)),
            lambda ws, out, slot, lengths: lib.avb_png_encode_u8(
                frames.data_ptr(), n, h, w, fs, rs, _fptr(header), int(header.size), out, slot, lengths, ws,
                eng.stream_ptr()), 10)
