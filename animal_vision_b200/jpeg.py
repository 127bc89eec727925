"""Device JPEG encode (K8, include/avb200.h avb_jpeg_encode_u8): the bytes of
`cv2.imencode(".jpg", frame, [cv2.IMWRITE_JPEG_QUALITY, quality])` for a batch of frames, computed on the GPU.
Only the compressed bytes cross to the host."""
from __future__ import annotations

from typing import List

import numpy as np

from . import tables
from ._abi import AvbError, check
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
        slot = int(lib.avb_jpeg_bound_bytes(h, w))
        need = int(lib.avb_jpeg_workspace_bytes(n, h, w))
        if slot <= 0 or need <= 0:
            check(min(slot, need), "avb_jpeg_workspace_bytes")
        key = ("jpeg", eng.stream_ptr())                    # per stream: encodes on different streams may overlap
        bufs = eng._cache.get(key)
        if bufs is None or bufs[0].numel() < need or bufs[1].numel() < n * slot or bufs[2].numel() < n:
            eng._cache[key] = None
            bufs = eng._cache[key] = (torch.empty(need, dtype=torch.uint8, device=eng.device),
                                      torch.empty(n * slot, dtype=torch.uint8, device=eng.device),
                                      torch.empty(n, dtype=torch.int64, device=eng.device))
        ws, out, lengths = bufs
        rc = lib.avb_jpeg_encode_u8(frames.data_ptr(), n, h, w, fs, rs, _fptr(header), int(header.size), _fptr(qt),
                                    out.data_ptr(), slot, lengths.data_ptr(), ws.data_ptr(), eng.stream_ptr())
        check(rc, "avb_jpeg_encode_u8")
        eng.launches += 7
        lens = lengths[:n].cpu().tolist()                   # waits for the encode
        offs = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
        host = torch.empty(int(offs[-1]), dtype=torch.uint8).pin_memory()
        for f in range(n):
            host[int(offs[f]):int(offs[f + 1])].copy_(out[f * slot:f * slot + lens[f]], non_blocking=True)
        torch.cuda.current_stream(eng.device).synchronize()
        buf = host.numpy().tobytes()
    return [buf[int(offs[f]):int(offs[f + 1])] for f in range(n)]
