"""ctypes binding of libavb200.so (include/avb200.h).

The library is built in-tree by `animal_vision_b200._build` (nvcc, sm_100a).  There is NO CPU
fallback: if the library cannot be built / loaded, or no CUDA device is present, every compute
entry point raises.
"""
from __future__ import annotations

import ctypes as C
import os
import threading
import warnings

from . import _build

_lock = threading.Lock()
_lib = None

AVB_VERSION = 170         # include/avb200.h AVB_VERSION
AVB_JPEG_HEADER_MAX = 1024
AVB_PNG_HEADER_LEN = 35
AVB_NORM_DIV255 = 0
AVB_NORM_AUTO = 1
AVB_ENC_TABLE_MAX = 2048
AVB_F32_POINT, AVB_F32_GAUSS, AVB_F32_STREAK = 0, 1, 2
AVB_IMG_NORM_UV, AVB_IMG_NORM_MAMMAL = 0, 1
AVB_STAT_MIN, AVB_STAT_MAX, AVB_STAT_MEAN = 0, 1, 2

_p = C.c_void_p
_i = C.c_int
_i64 = C.c_int64
_f = C.c_float

# name -> (restype, argtypes); must list every symbol include/avb200.h declares
SIGNATURES = {
    "avb_version": (_i, []),
    "avb_last_error": (C.c_char_p, []),
    "avb_header_sha": (C.c_char_p, []),
    "avb_profile_begin": (_i, []),
    "avb_profile_end": (_i, [_p, _i, _p, _i]),
    "avb_build_encode_table": (_i, [_p, _p, _i]),
    "avb_colorimetric_u8": (_i, [_p, _p, _i, _i, _i, _i64, _i64, _i64, _i64, _p, _p, _p, _p, _p, _i, _p, _p]),
    "avb_dichromat_blur_u8": (_i, [_p, _p, _i, _i, _i, _i64, _i64, _i64, _i64, _p, _p, _p, _p, _p, _i, _i, _p, _p]),
    "avb_streak_blur_u8": (_i, [_p, _p, _i, _i, _i, _i64, _i64, _i64, _i64, _p, _p, _p, _p, _f, _i, _p, _p]),
    "avb_cat_u8": (_i, [_p, _p, _p, _i, _i, _i, _i64, _i64, _i64, _i64, _i64, _i64, _p, _p, _p, _p, _p, _i, _p, _p, _i, _p, _p]),
    "avb_mstpp_create": (_i, [_p, _i64, _p]),
    "avb_mstpp_destroy": (_i, [_p]),
    "avb_mstpp_workspace_bytes": (_i64, [_i, _i, _i, _i, _i]),
    "avb_mstpp_forward": (_i, [_p, _p, _i, _p, _i, _i, _i, _i, _i, _p, _p]),
    "avb_mstpp_forward_bands": (_i, [_p, _p, _i, _p, _p, _p, _i, _i, _i, _i, _i, _i, _p, _p]),
    "avb_band_project_f32": (_i, [_p, _p, _p, _i64, _i, _i, _p]),
    "avb_safe_norm_f32": (_i, [_p, _p, _i64, _i, _i, _p, _p]),
    "avb_dichromat_f32": (_i, [_p, _p, _p, _i, _i, _i, _p, _i, _p, _i, _p, _p, _f, _i, _p, _p]),
    "avb_img_to_float01": (_i, [_p, _i, _p, _i, _i64, _i, _p, _p]),
    "avb_img_resample": (_i, [_p, _p, _i, _i, _i, _i, _i, _i64, _i64, _p, _p, _i, _p]),
    "avb_img_blur": (_i, [_p, _p, _p, _i, _i, _i, _i, _p, _i, _p, _i, _p]),
    "avb_img_stats": (_i, [_p, _i, _i64, _i, _p, _p, _p]),
    "avb_img_divide_channels": (_i, [_p, _p, _i, _i64, _i, _p, _i, _f, _p]),
    "avb_img_percentile_scratch_bytes": (_i64, [_i]),
    "avb_img_percentile": (_i, [_p, _i64, _i64, _p, _p, _i, _p, _p, _p]),
    "avb_cat_warp_f32": (_i, [_p, _p, _i, _i, _i, _p, _p]),
    "avb_uv_catches_f32": (_i, [_p, _p, _i64, _p, _p, _i, _f, _p]),
    "avb_uv_map_f32": (_i, [_p, _p, _i, _i, _i, _i, _i, _i64, _i64, _p, _i, _p, _f, _p, _p]),
    "avb_uv_workspace_bytes": (_i64, [_i, _i, _i, _i]),
    "avb_vm_run": (_i, [_p, _i, _i, _i, _i, _i, _p, _i, _p, _i, _p]),
    "avb_img_remap": (_i, [_p, _p, _i, _i, _i, _i, _p, _p, _p]),
    "avb_uv_map_u8": (_i, [_p, _p, _i, _i, _i, _i64, _i64, _i64, _i64, _p, _p, _p, _p, _i, _f, _i, _p, _i, _i, _p, _f, _p, _p, _p]),
    "avb_jpeg_bound_bytes": (_i64, [_i, _i]),
    "avb_jpeg_workspace_bytes": (_i64, [_i, _i, _i]),
    "avb_jpeg_encode_u8": (_i, [_p, _i, _i, _i, _i64, _i64, _p, _i, _p, _p, _i64, _p, _p, _p]),
    "avb_jpeg_encode_rgb_u8": (_i, [_p, _i, _i, _i, _i64, _i64, _p, _i, _p, _p, _i64, _p, _p, _p]),
    "avb_jpeg_opt_workspace_bytes": (_i64, [_i, _i, _i]),
    "avb_jpeg_opt_encode_u8": (_i, [_p, _i, _i, _i, _i64, _i64, _p, _i, _p, _i, _p, _p, _i64, _p, _p, _p]),
    "avb_jpeg_opt_encode_rgb_u8": (_i, [_p, _i, _i, _i, _i64, _i64, _p, _i, _p, _i, _p, _p, _i64, _p, _p, _p]),
    "avb_mjpeg_pack_u8": (_i, [_p, _i64, _p, _i, _p, _p, _p]),
    "avb_png_bound_bytes": (_i64, [_i, _i]),
    "avb_png_workspace_bytes": (_i64, [_i, _i, _i]),
    "avb_png_encode_u8": (_i, [_p, _i, _i, _i, _i64, _i64, _p, _i, _p, _i64, _p, _p, _p]),
    "avb_split_compose_u8": (_i, [_p, _p, _p, _i, _i, _i, _i64, _i64, _i64, _i64, _i64, _i64, _i, _i, _p, _p, _p]),
    "avb_split_fetch_u8": (_i, [_p, _p, _i, _i, _i, _i64, _i64, _i64, _i64, _i, _p]),
}


class AvbError(RuntimeError):
    pass


def lib_path() -> str:
    return _build.LIB


def load(build_if_missing: bool = True) -> C.CDLL:
    """Load (building first if the sources changed) and type every exported symbol."""
    global _lib
    with _lock:
        if _lib is not None:
            return _lib
        path = _build.LIB
        if build_if_missing and not _build.is_current():
            try:
                _build.build()
            except Exception as e:
                # a stale binary is only used on explicit request, and never if its ABI differs (checked below)
                if not os.path.exists(path):
                    raise AvbError(f"libavb200.so is missing and could not be built: {e}") from e
                if os.environ.get("AVB_ALLOW_STALE_LIB") != "1":
                    raise AvbError(f"libavb200.so is out of date and the rebuild failed ({e}); set AVB_ALLOW_STALE_LIB=1 "
                                   "to load the stale binary anyway") from e
                warnings.warn(f"loading a STALE libavb200.so (rebuild failed: {e})", RuntimeWarning)
        if not os.path.exists(path):
            raise AvbError(f"{path} not found: run `python -m animal_vision_b200._build` (no CPU fallback exists)")
        lib = C.CDLL(path)
        try:
            sha_fn = lib.avb_header_sha
            sha_fn.restype = C.c_char_p
            built_against = sha_fn().decode()
        except AttributeError:
            built_against = "absent"
        if built_against != _build.header_sha():
            raise AvbError(f"{path} was compiled against another include/avb200.h (library {built_against}, header "
                           f"{_build.header_sha()}): rebuild with `python -m animal_vision_b200._build --force`")
        if int(lib.avb_version()) != AVB_VERSION:
            raise AvbError(f"{path}: avb_version() = {int(lib.avb_version())}, binding expects {AVB_VERSION}")
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)          # AttributeError if the .so does not export it
            fn.restype = res
            fn.argtypes = args
        _lib = lib
        return lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = load().avb_last_error().decode(errors="replace")
        raise AvbError(f"{what} failed (rc={rc}): {msg}")
