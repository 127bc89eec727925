"""Device JPEG encode (K8, include/avb200.h avb_jpeg_encode_u8): the bytes of
`cv2.imencode(".jpg", frame, [cv2.IMWRITE_JPEG_QUALITY, quality])` for a batch of frames, computed on the GPU.
Only the compressed bytes cross to the host."""
from __future__ import annotations

from typing import List

import numpy as np

from . import tables
from ._abi import AvbError
from ._slots import encode_slots
from .engine import _fptr, get_engine


def encode_jpeg(frames, quality: int = 95) -> List[bytes]:
    """frames: CUDA uint8 tensor [N,H,W,3] in the channel order cv2.imencode expects (BGR), packed pixels, any row
    and frame strides.  Runs on the current stream; returns one JPEG file per frame."""
    import torch
    if not (isinstance(frames, torch.Tensor) and frames.is_cuda):
        raise AvbError("encode_jpeg: expected a CUDA uint8 tensor [N,H,W,3]")
    if isinstance(quality, bool) or not isinstance(quality, (int, np.integer)) or not 1 <= int(quality) <= 100:
        raise AvbError(f"encode_jpeg: quality must be an integer in [1, 100], got {quality!r}")
    eng = get_engine(frames.device)
    n, h, w, fs, rs = eng.check_frames(frames)
    if n == 0:
        return []
    if not (1 <= h <= 65535 and 1 <= w <= 65535):
        raise AvbError(f"encode_jpeg: frame size {h}x{w} outside [1, 65535]^2")
    header = np.frombuffer(tables.jpeg_header(h, w, int(quality)), np.uint8)
    qt = np.ascontiguousarray(tables.jpeg_quant_tables(int(quality)))
    with torch.cuda.device(eng.device):
        lib = eng.lib
        return encode_slots(
            eng, "jpeg", n, int(lib.avb_jpeg_bound_bytes(h, w)), int(lib.avb_jpeg_workspace_bytes(n, h, w)),
            lambda ws, out, slot, lengths: lib.avb_jpeg_encode_u8(
                frames.data_ptr(), n, h, w, fs, rs, _fptr(header), int(header.size), _fptr(qt), out, slot, lengths, ws,
                eng.stream_ptr()), 7)
