"""Motion-JPEG AVI writer (host only): the container `cv2.VideoWriter(path, cv2.CAP_OPENCV_MJPEG, fourcc("MJPG"), fps,
size)` writes, filled with JPEG files encoded elsewhere, typically on the device by `HostBatchPipeline.run_split_jpeg`
(K8 + K11), which hands over whole chunks of frames as ready-made '00dc' records.

Layout, byte for byte that of OpenCV's writer (videoio container_avi.cpp): 'RIFF' 'AVI ', the 'hdrl' list ('avih', 'strl'
with 'strh' / 'strf', 'odml' with 'dmlh'), a 'JUNK' chunk up to the 'movi' list at offset 4096 (its fourcc at 4104), the
'00dc' records, then 'idx1' (flags AVIIF_KEYFRAME, offsets from the 'movi' fourcc).  The frame counts and the RIFF and
'movi' sizes are patched on close()."""
from __future__ import annotations

import struct
from typing import Sequence

RIFF_MAX = 2 ** 32 - 1          # the RIFF size field is a u32; OpenDML 'AVIX' continuation is not written
JUNK_END = 4096                 # the 'movi' list starts here, as in OpenCV's writer
MAX_BYTES_PER_SEC = 99999999
AVIF_FLAGS = 0x910              # AVIF_HASINDEX | AVIF_ISINTERLEAVED | AVIF_TRUSTCKTYPE
SUGGESTED_BUFFER = 1 << 20
AVIIF_KEYFRAME = 0x10
_FRAME_COUNT_AT = (48, 140, 232)   # avih dwTotalFrames, strh dwLength, dmlh dwTotalFrames
_MOVI_AT = JUNK_END + 4            # the 'movi' list's size field


def jpeg_record(jpeg: bytes) -> bytes:
    """The '00dc' chunk of one JPEG: fourcc, little-endian u32 size, the JPEG, zero bytes up to a multiple of 4 (the size
    counts them)."""
    pad = -len(jpeg) & 3
    return b"00dc" + struct.pack("<I", len(jpeg) + pad) + bytes(jpeg) + b"\0" * pad


def _chunk(fourcc: bytes, data: bytes) -> bytes:
    return fourcc + struct.pack("<I", len(data)) + data


def _list(kind: bytes, data: bytes) -> bytes:
    return _chunk(b"LIST", kind + data)


def avi_header(fps: float, width: int, height: int) -> bytes:
    """Everything before the 'movi' list, with frame counts 0: 4096 bytes."""
    rate = int(round(fps))
    us = int(round(1e6 / rate))
    avih = struct.pack("<14I", us, MAX_BYTES_PER_SEC, 0, AVIF_FLAGS, 0, 0, 1, SUGGESTED_BUFFER, width, height, 0, 0, 0, 0)
    strh = (b"vidsMJPG" + struct.pack("<IHHIIIIIIiI", 0, 0, 0, 0, 1, rate, 0, 0, SUGGESTED_BUFFER, -1, 0)
            + struct.pack("<4H", 0, 0, width, height))
    strf = struct.pack("<IiiHH4sIiiII", 40, width, height, 1, 24, b"MJPG", width * height * 3, 0, 0, 0, 0)
    hdrl = _list(b"hdrl", _chunk(b"avih", avih) + _list(b"strl", _chunk(b"strh", strh) + _chunk(b"strf", strf))
                 + _list(b"odml", _chunk(b"dmlh", struct.pack("<2I", 0, 0))))
    head = b"RIFF" + struct.pack("<I", 0) + b"AVI " + hdrl
    junk = _chunk(b"JUNK", bytes(JUNK_END - len(head) - 8))
    return head + junk


class MjpegAviWriter:
    """Writes a Motion-JPEG AVI at `path`: `fps` (stored as round(fps), as OpenCV does) and `size` = (width, height) as
    cv2.VideoWriter takes them.  `write_records` appends ready-made '00dc' records (run_split_jpeg's `out`),
    `write_jpeg` one JPEG file.

    The whole file is one RIFF, so it stays below 2**32 - 1 bytes, index included: about 1 600 4K frames at quality 95.
    A record that would cross that raises ValueError before any of its bytes are written; the records before it stay,
    and close() still leaves a valid AVI.  Use as a context manager or call close()."""

    def __init__(self, path, fps: float, size: Sequence[int]):
        width, height = (int(v) for v in size)
        if not (1 <= width <= 65535 and 1 <= height <= 65535):
            raise ValueError(f"MjpegAviWriter: size {tuple(size)} outside [1, 65535]^2")
        if not fps > 0 or int(round(fps)) < 1:
            raise ValueError(f"MjpegAviWriter: fps must round to a positive integer, got {fps!r}")
        self.path = path
        self.fps, self.size = fps, (width, height)
        self._fh = open(path, "wb")
        self._fh.write(avi_header(fps, width, height))
        self._fh.write(b"LIST" + struct.pack("<I", 0) + b"movi")
        self._pos = JUNK_END + 12           # file size so far
        self._index = bytearray()
        self.frames = 0

    def write_jpeg(self, jpeg: bytes) -> None:
        """Append one JPEG file as a frame."""
        self.write_records(memoryview(jpeg_record(jpeg)), [len(jpeg)])

    def write_records(self, records, jpeg_lengths: Sequence[int]) -> None:
        """Append consecutive '00dc' records (bytes-like), one per frame, of JPEGs `jpeg_lengths` bytes long."""
        if self._fh is None:
            raise ValueError("MjpegAviWriter: write to a closed writer")
        mv = memoryview(records).cast("B")
        sizes = [(int(n) + 3) & ~3 for n in jpeg_lengths]
        if 8 * len(sizes) + sum(sizes) != mv.nbytes:
            raise ValueError(f"MjpegAviWriter: {mv.nbytes} record bytes for JPEGs of {list(jpeg_lengths)} bytes")
        off = 0
        for k, size in enumerate(sizes):
            if bytes(mv[off:off + 4]) != b"00dc" or struct.unpack_from("<I", mv, off + 4)[0] != size:
                raise ValueError(f"MjpegAviWriter: record {k} is not a '00dc' chunk of {size} bytes")
            # the file after this record and an index of every frame so far, less the RIFF fourcc and size
            if self._pos + off + 8 + size + 8 + 16 * (self.frames + k + 1) - 8 > RIFF_MAX:
                self._append(mv[:off], sizes[:k])
                raise ValueError(f"MjpegAviWriter: frame {self.frames} would take the file past the AVI limit of "
                                 f"{RIFF_MAX} bytes (OpenDML is not written); {self.frames} frames are kept")
            off += 8 + size
        self._append(mv, sizes)

    def _append(self, mv: memoryview, sizes: Sequence[int]) -> None:
        off = self._pos - _MOVI_AT - 4          # from the 'movi' fourcc
        for size in sizes:
            self._index += b"00dc" + struct.pack("<3I", AVIIF_KEYFRAME, off, size)
            off += 8 + size
        self._fh.write(mv)
        self._pos += mv.nbytes
        self.frames += len(sizes)

    def close(self) -> None:
        """Write the index and patch the sizes and frame counts."""
        if self._fh is None:
            return
        fh, self._fh = self._fh, None
        try:
            fh.write(_chunk(b"idx1", bytes(self._index)))
            end = self._pos + 8 + len(self._index)
            for at, value in [(4, end - 8), (_MOVI_AT, self._pos - _MOVI_AT - 4)] + \
                    [(at, self.frames) for at in _FRAME_COUNT_AT]:
                fh.seek(at)
                fh.write(struct.pack("<I", value))
        finally:
            fh.close()

    def __enter__(self) -> "MjpegAviWriter":
        return self

    def __exit__(self, *exc) -> None:
        self.close()
