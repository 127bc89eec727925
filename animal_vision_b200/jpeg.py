"""Device JPEG encode (K8, include/avb200.h avb_jpeg_encode_u8 / avb_jpeg_encode_rgb_u8): the bytes of
`cv2.imencode(".jpg", frame, [cv2.IMWRITE_JPEG_QUALITY, quality])` for a batch of frames, computed on the GPU; with
`optimize=True` (avb_jpeg_opt_encode_u8 / avb_jpeg_opt_encode_rgb_u8) the bytes of the same call with
`cv2.IMWRITE_JPEG_OPTIMIZE`, Huffman tables built on the device from each frame's own symbol counts.  Only the compressed
bytes cross to the host."""
from __future__ import annotations

from typing import List

import numpy as np

from . import tables
from ._abi import AvbError
from ._slots import encode_slots
from .engine import _fptr, get_engine


JPEG_LAUNCHES = 7                 # kernels one K8 encode launches (csrc/k8_jpeg.cu)
JPEG_OPT_LAUNCHES = 11            # kernels (10) and memsets (1) one optimized K8 encode launches


def check_quality(quality, what: str = "encode_jpeg") -> int:
    if isinstance(quality, bool) or not isinstance(quality, (int, np.integer)) or not 1 <= int(quality) <= 100:
        raise AvbError(f"{what}: quality must be an integer in [1, 100], got {quality!r}")
    return int(quality)


class JpegLauncher:
    """K8 for frames of one shape and quality: the header (or, optimized, the header prefix and SOS) and quantiser
    tables built once, the sizes of the slots and the workspace, and `launch` of n frames on the current stream."""

    def __init__(self, lib, h: int, w: int, quality: int, rgb: bool, optimize: bool = False):
        if not (1 <= h <= 65535 and 1 <= w <= 65535):
            raise AvbError(f"encode_jpeg: frame size {h}x{w} outside [1, 65535]^2")
        self.lib, self.h, self.w, self.optimize = lib, h, w, bool(optimize)
        self.qt = np.ascontiguousarray(tables.jpeg_quant_tables(quality))
        self.slot = int(lib.avb_jpeg_bound_bytes(h, w))
        if self.optimize:
            self.header = np.frombuffer(tables.jpeg_header_prefix(h, w, quality), np.uint8)
            self.sos = np.frombuffer(tables.JPEG_SOS, np.uint8)
            self.name = "avb_jpeg_opt_encode_rgb_u8" if rgb else "avb_jpeg_opt_encode_u8"
            self.launches = JPEG_OPT_LAUNCHES
        else:
            self.header = np.frombuffer(tables.jpeg_header(h, w, quality), np.uint8)
            self.name = "avb_jpeg_encode_rgb_u8" if rgb else "avb_jpeg_encode_u8"
            self.launches = JPEG_LAUNCHES
        self.fn = getattr(lib, self.name)

    def workspace_bytes(self, n: int) -> int:
        fn = self.lib.avb_jpeg_opt_workspace_bytes if self.optimize else self.lib.avb_jpeg_workspace_bytes
        return int(fn(n, self.h, self.w))

    def launch(self, frames_ptr: int, n: int, fs: int, rs: int, ws: int, out: int, slot: int, lengths: int,
               stream: int) -> int:
        if self.optimize:
            return self.fn(frames_ptr, n, self.h, self.w, fs, rs, _fptr(self.header), int(self.header.size),
                           _fptr(self.sos), int(self.sos.size), _fptr(self.qt), out, slot, lengths, ws, stream)
        return self.fn(frames_ptr, n, self.h, self.w, fs, rs, _fptr(self.header), int(self.header.size), _fptr(self.qt),
                       out, slot, lengths, ws, stream)


def encode_jpeg(frames, quality: int = 95, *, rgb: bool = False, optimize: bool = False) -> List[bytes]:
    """frames: CUDA uint8 tensor [N,H,W,3] in the channel order cv2.imencode expects (BGR), or in RGB order with
    `rgb=True` (the bytes of cv2.imencode of `frame[..., ::-1]`); packed pixels, any row and frame strides.  With
    `optimize=True` each file has Huffman tables built from its frame's symbol counts (cv2.IMWRITE_JPEG_OPTIMIZE): the
    same pixels, usually fewer bytes.  Runs on the current stream; returns one JPEG file per frame."""
    import torch
    if not (isinstance(frames, torch.Tensor) and frames.is_cuda):
        raise AvbError("encode_jpeg: expected a CUDA uint8 tensor [N,H,W,3]")
    quality = check_quality(quality)
    eng = get_engine(frames.device)
    n, h, w, fs, rs = eng.check_frames(frames)
    if n == 0:
        return []
    k8 = JpegLauncher(eng.lib, h, w, quality, bool(rgb), bool(optimize))
    with torch.cuda.device(eng.device):
        return encode_slots(
            eng, "jpeg_opt" if k8.optimize else "jpeg", n, k8.slot, k8.workspace_bytes(n),
            lambda ws, out, slot, lengths: k8.launch(frames.data_ptr(), n, fs, rs, ws, out, slot, lengths,
                                                     eng.stream_ptr()), k8.launches)
