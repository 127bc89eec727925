"""Per-device engine: owns the device-resident tables, scratch and the pinned staging buffers of
the NumPy compatibility shim, and wraps each C-ABI entry point for torch tensors.

Host code is plumbing only (torch for device memory and streams); all pixel work happens in
libavb200.so.  No CPU fallback: constructing an Engine without a CUDA device raises.
"""
from __future__ import annotations

import ctypes as C
import functools
import threading
from typing import Dict, Tuple

import numpy as np

from . import _abi, tables
from ._abi import AVB_NORM_AUTO, AVB_NORM_DIV255, AvbError, check

_engines: Dict[int, "Engine"] = {}
_engines_lock = threading.Lock()


def get_engine(device=None) -> "Engine":
    import torch
    if not torch.cuda.is_available():
        raise AvbError("animal_vision_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
    idx = torch.cuda.current_device() if device is None else torch.device(device).index or 0
    with _engines_lock:
        if idx not in _engines:
            _engines[idx] = Engine(idx)
        return _engines[idx]


def split_fetch_bytes(n: int, h: int, w: int, band_rows: int) -> int:
    """Bytes Engine.split_fetch copies for n frames of h x w: the label band whole, then columns [w // 2, w)."""
    return n * (band_rows * 3 * w + (h - band_rows) * (3 * w - 3 * (w // 2)))


def _fptr(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)


def _on_device(fn):
    """Run an Engine method with the engine's device current: kernel launches, sm_count() and the
    per-device shared-memory opt-in all act on the CURRENT device, the stream belongs to self.device."""
    @functools.wraps(fn)
    def wrapper(self, *a, **kw):
        with self.torch.cuda.device(self.device):
            return fn(self, *a, **kw)
    return wrapper


class Engine:
    def __init__(self, device_index: int):
        import torch
        self.torch = torch
        self.lib = _abi.load()
        self.device = torch.device("cuda", device_index)
        with torch.cuda.device(self.device):
            self.dec = self._dev(tables.decode_lut(True))
            self.dec_raw = self._dev(tables.decode_lut(False))
            self.dec_torch = self._dev(tables.decode_lut_torch())
            self.enc = self._dev(self._encode_table(tables.encode_thresholds(False)))
            self.enc64 = self._dev(self._encode_table(tables.encode_thresholds(True)))
        self._cache: Dict[Tuple, object] = {}
        self._flags = None
        self._staging: Dict[Tuple, Tuple] = {}
        self.launches = 0          # kernels launched through this engine (bench.py reports it)

    # ------------------------------------------------------------------ helpers
    def _dev(self, a: np.ndarray):
        return self.torch.from_numpy(np.ascontiguousarray(a).copy()).to(self.device)

    def _encode_table(self, thr: np.ndarray) -> np.ndarray:
        buf = np.zeros(_abi.AVB_ENC_TABLE_MAX, np.uint32)
        n = self.lib.avb_build_encode_table(_fptr(np.ascontiguousarray(thr, np.float32)), _fptr(buf), buf.size)
        if n <= 0:
            check(n, "avb_build_encode_table")
        return buf[:n].view(np.int32)      # torch has no uint32 arithmetic; bits are what matter

    def cached(self, key, build):
        v = self._cache.get(key)
        if v is None:
            v = self._cache[key] = build()
        return v

    def flags(self, n: int):
        """Per-frame flag / scratch words.  One buffer PER STREAM: batches of different species may run
        concurrently on different streams and must not share scratch."""
        key = self.stream_ptr()
        if self._flags is None:
            self._flags = {}
        buf = self._flags.get(key)
        if buf is None or buf.numel() < n:
            buf = self._flags[key] = self.torch.zeros(max(n, 64), dtype=self.torch.int32, device=self.device)
        return buf

    def stream_ptr(self) -> int:
        return self.torch.cuda.current_stream(self.device).cuda_stream

    def check_frames(self, frames, name="frames"):
        t = self.torch
        if not (isinstance(frames, t.Tensor) and frames.is_cuda and frames.dtype == t.uint8 and frames.dim() == 4
                and frames.shape[3] == 3 and frames.stride(3) == 1 and frames.stride(2) == 3):
            raise AvbError(f"{name}: expected a CUDA uint8 tensor [N,H,W,3] with packed pixels")
        if frames.device != self.device:
            raise AvbError(f"{name} lives on {frames.device}, engine on {self.device}")
        n, h, w, _ = frames.shape
        return n, h, w, frames.stride(0), frames.stride(1)

    # ------------------------------------------------------------------ C-ABI wrappers
    @_on_device
    def colorimetric(self, frames, out, M: np.ndarray, row_gain=None, norm=AVB_NORM_AUTO):
        n, h, w, fs, rs = self.check_frames(frames)
        _, _, _, ofs, ors = self.check_frames(out, "out")
        M = np.ascontiguousarray(M, np.float32)
        rc = self.lib.avb_colorimetric_u8(
            frames.data_ptr(), out.data_ptr(), n, h, w, fs, rs, ofs, ors,
            self.dec.data_ptr(), self.dec_raw.data_ptr(), self.enc.data_ptr(), _fptr(M),
            None if row_gain is None else row_gain.data_ptr(), norm,
            self.flags(n).data_ptr() if norm == AVB_NORM_AUTO else None, self.stream_ptr())
        check(rc, "avb_colorimetric_u8")
        self.launches += 2 if norm == AVB_NORM_AUTO else 1

    @_on_device
    def dichromat_blur(self, frames, out, M: np.ndarray, taps: np.ndarray, norm=AVB_NORM_AUTO):
        n, h, w, fs, rs = self.check_frames(frames)
        _, _, _, ofs, ors = self.check_frames(out, "out")
        M = np.ascontiguousarray(M, np.float32)
        taps = np.ascontiguousarray(taps, np.float32)
        rc = self.lib.avb_dichromat_blur_u8(
            frames.data_ptr(), out.data_ptr(), n, h, w, fs, rs, ofs, ors,
            self.dec.data_ptr(), self.dec_raw.data_ptr(), self.enc.data_ptr(), _fptr(M), _fptr(taps), int(taps.size),
            norm, self.flags(n).data_ptr() if norm == AVB_NORM_AUTO else None, self.stream_ptr())
        check(rc, "avb_dichromat_blur_u8")
        self.launches += 2 if norm == AVB_NORM_AUTO else 1

    @_on_device
    def streak_blur(self, frames, out, M: np.ndarray, streak, chroma: float = 0.0, norm=AVB_NORM_AUTO):
        n, h, w, fs, rs = self.check_frames(frames)
        _, _, _, ofs, ors = self.check_frames(out, "out")
        M = np.ascontiguousarray(M, np.float32)
        key = ("streak", h, M.tobytes(), tuple(float(v) for v in streak))
        tab = self.cached(key, lambda: self._dev(tables.streak_row_table(h, M, *streak)))
        rc = self.lib.avb_streak_blur_u8(
            frames.data_ptr(), out.data_ptr(), n, h, w, fs, rs, ofs, ors,
            self.dec.data_ptr(), self.dec_raw.data_ptr(), self.enc.data_ptr(), tab.data_ptr(), float(chroma),
            norm, self.flags(n).data_ptr() if norm == AVB_NORM_AUTO else None, self.stream_ptr())
        check(rc, "avb_streak_blur_u8")
        self.launches += 2 if norm == AVB_NORM_AUTO else 1

    @_on_device
    def dichromat_f32(self, frames, out, tmp, M: np.ndarray, kind: int, taps=None, streak=None, row_gain=None,
                      chroma: float = 0.0, quantize: bool = False):
        """Float-frame path (include/avb200.h avb_dichromat_f32): packed float32 CUDA tensors [N,H,W,3]."""
        t = self.torch
        for name, x in (("frames", frames), ("out", out), ("tmp", tmp)):
            if not (x.is_cuda and x.dtype == t.float32 and x.dim() == 4 and x.shape[3] == 3 and x.is_contiguous()):
                raise AvbError(f"{name} must be a contiguous float32 CUDA tensor [N,H,W,3]")
        n, h, w, _ = frames.shape
        M = np.ascontiguousarray(M, np.float32)
        tab = None
        if streak is not None:
            key = ("streak", h, M.tobytes(), tuple(float(v) for v in streak))
            tab = self.cached(key, lambda: self._dev(tables.streak_row_table(h, M, *streak)))
        tp = None if taps is None else np.ascontiguousarray(taps, np.float32)
        rc = self.lib.avb_dichromat_f32(
            frames.data_ptr(), out.data_ptr(), tmp.data_ptr(), n, h, w, _fptr(M), kind,
            None if tp is None else _fptr(tp), 0 if tp is None else int(tp.size),
            None if tab is None else tab.data_ptr(), None if row_gain is None else row_gain.data_ptr(),
            float(chroma), int(bool(quantize)), self.flags(n).data_ptr(), self.stream_ptr())
        check(rc, "avb_dichromat_f32")
        self.launches += 3 + (kind != 0) + (kind == 1)

    @_on_device
    def cat(self, frames, out_human, out_cat, M: np.ndarray, taps: np.ndarray, warp_dev, zoom_dev, norm=AVB_NORM_AUTO):
        n, h, w, fs, rs = self.check_frames(frames)
        _, _, _, hfs, hrs = self.check_frames(out_human, "out_human")
        _, _, _, cfs, crs = self.check_frames(out_cat, "out_cat")
        M = np.ascontiguousarray(M, np.float32)
        taps = np.ascontiguousarray(taps, np.float32)
        rc = self.lib.avb_cat_u8(
            frames.data_ptr(), out_human.data_ptr(), out_cat.data_ptr(), n, h, w, fs, rs, hfs, hrs, cfs, crs,
            self.dec.data_ptr(), self.dec_raw.data_ptr(),
            self.enc64.data_ptr(), _fptr(M), _fptr(taps), int(taps.size),
            None if warp_dev is None else warp_dev.data_ptr(), zoom_dev.data_ptr(),
            norm, self.flags(n).data_ptr() if norm == AVB_NORM_AUTO else None, self.stream_ptr())
        check(rc, "avb_cat_u8")
        self.launches += 3 if norm == AVB_NORM_AUTO else 2

    @_on_device
    def uv_map(self, frames, out, M3: np.ndarray, bands_dev, denom_eps: float, adapt_mode: int,
               blur_taps: np.ndarray, map_mode: int = 0, map_params=None, mix_alpha: float = 0.45, dbg_catches=None):
        n, h, w, fs, rs = self.check_frames(frames)
        _, _, _, ofs, ors = self.check_frames(out, "out")
        need = int(self.lib.avb_uv_workspace_bytes(n, h, w, int(map_mode)))
        if need <= 0:
            raise AvbError("avb_uv_workspace_bytes: bad arguments")
        ws_key = ("uv_ws", self.stream_ptr())                 # per stream, like flags()
        ws = self._cache.get(ws_key)
        if ws is None or ws.numel() < need:
            self._cache[ws_key] = None
            ws = self._cache[ws_key] = self.torch.empty(need, dtype=self.torch.uint8, device=self.device)
        M3 = np.ascontiguousarray(M3, np.float32)
        taps = np.ascontiguousarray(blur_taps, np.float32)
        mp = None if map_params is None else np.ascontiguousarray(map_params, np.float32)
        assert mp is None or mp.size == 15
        rc = self.lib.avb_uv_map_u8(
            frames.data_ptr(), out.data_ptr(), n, h, w, fs, rs, ofs, ors,
            self.dec_torch.data_ptr(), self.enc.data_ptr(), _fptr(M3),
            None if bands_dev is None else bands_dev.data_ptr(), 0 if bands_dev is None else int(bands_dev.shape[0]),
            float(denom_eps), int(adapt_mode), _fptr(taps) if taps.size else None, int(taps.size),
            int(map_mode), None if mp is None else _fptr(mp), float(mix_alpha),
            ws.data_ptr(), None if dbg_catches is None else dbg_catches.data_ptr(), self.stream_ptr())
        check(rc, "avb_uv_map_u8")
        self.launches += 3 + (4 if map_mode != 2 else 0)      # stats, prep, [hist, scan, collect, select], map

    def split_stencil(self, h: int, w: int, left: str, right: str):
        """(band_rows, class map, tables) of the corner labels of an h x w split frame on this device
        (tables.split_label_stencil), built and uploaded once per (h, w, labels)."""
        def build():
            st = tables.split_label_stencil(int(h), int(w), str(left), str(right))
            with self.torch.cuda.device(self.device):
                return st.band_rows, self._dev(st.classes.view(np.int16)), self._dev(st.luts)
        return self.cached(("split_labels", int(h), int(w), str(left), str(right)), build)

    @_on_device
    def split_compose(self, left, right, out, seam: bool, stencil=None):
        """K9 (avb_split_compose_u8) on the current stream: `out` = left half of `left`, right half of `right`, the seam,
        and the labels of `stencil` (from split_stencil; None for none)."""
        n, h, w, lfs, lrs = self.check_frames(left, "original")
        _, _, _, rfs, rrs = self.check_frames(right, "modified")
        _, _, _, ofs, ors = self.check_frames(out, "out")
        if n == 0 or h == 0 or w == 0:
            return
        band, cls, lut = stencil if stencil is not None else (0, None, None)
        rc = self.lib.avb_split_compose_u8(
            left.data_ptr(), right.data_ptr(), out.data_ptr(), n, h, w, lfs, lrs, rfs, rrs, ofs, ors, int(seam), band,
            None if cls is None else cls.data_ptr(), None if lut is None else lut.data_ptr(), self.stream_ptr())
        check(rc, "avb_split_compose_u8")
        self.launches += 1

    @_on_device
    def split_fetch(self, src, dst, band_rows: int) -> int:
        """avb_split_fetch_u8 on the current stream: copy into the page-locked host frames `dst` the bytes of the composed
        split frames `src` (CUDA, same shape) that can differ from the input frames -- rows [0, band_rows) and the columns
        [W // 2, W) of the other rows.  With `dst` holding the frames `src` was composed from, `dst` becomes the split
        frames.  Returns the bytes copied (split_fetch_bytes)."""
        n, h, w, sfs, srs = self.check_frames(src, "src")
        t = self.torch
        if not (isinstance(dst, t.Tensor) and dst.device.type == "cpu" and dst.dtype == t.uint8
                and tuple(dst.shape) == (n, h, w, 3) and dst.stride(3) == 1 and dst.stride(2) == 3):
            raise AvbError("dst: expected a host uint8 tensor of src's shape with packed pixels")
        if n == 0 or h == 0 or w == 0:
            return 0
        rc = self.lib.avb_split_fetch_u8(src.data_ptr(), dst.data_ptr(), n, h, w, sfs, srs, dst.stride(0), dst.stride(1),
                                         int(band_rows), self.stream_ptr())
        check(rc, "avb_split_fetch_u8")
        return split_fetch_bytes(n, h, w, band_rows)

    # ------------------------------------------------------------------ NumPy shim staging
    @_on_device
    def staging(self, shape, slots: int = 1):
        """(pinned_in, dev_in, [dev_out...], [pinned_out...]) for one HxWx3 uint8 frame."""
        key = (tuple(shape), slots, threading.get_ident())     # one buffer set per calling thread: visualize() is re-entrant
        s = self._staging.get(key)
        if s is None:
            t = self.torch
            pin_in = t.empty((1,) + tuple(shape), dtype=t.uint8).pin_memory()
            dev_in = t.empty((1,) + tuple(shape), dtype=t.uint8, device=self.device)
            dev_out = [t.empty((1,) + tuple(shape), dtype=t.uint8, device=self.device) for _ in range(slots)]
            pin_out = [t.empty((1,) + tuple(shape), dtype=t.uint8).pin_memory() for _ in range(slots)]
            s = self._staging[key] = (pin_in, dev_in, dev_out, pin_out)
        return s
