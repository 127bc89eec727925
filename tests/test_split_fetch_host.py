"""The split-frame fetch on the CPU: the argument checks of avb_split_fetch_u8 that fail before any CUDA call, and the
byte set it copies -- exactly where a labelled split frame can differ from its input, counted by split_fetch_bytes."""
import numpy as np
import pytest
import torch

import frames
from animal_vision_b200 import tables
from animal_vision_b200.engine import split_fetch_bytes
from animal_vision_b200.renderers.video import draw_split_labels, split_compare_batch


def fetch_mask(h, w, band_rows):
    """[h, 3w] bool: the bytes of one frame that avb_split_fetch_u8 copies."""
    m = np.zeros((h, 3 * w), bool)
    m[:band_rows] = True
    m[band_rows:, 3 * (w // 2):] = True
    return m


@pytest.mark.parametrize("h,w,band", [(1, 1, 0), (1, 1, 1), (5, 1, 5), (5, 1, 0), (2, 3, 1), (9, 13, 9), (135, 241, 41),
                                      (1080, 1920, 67), (1079, 1921, 0), (2160, 3840, 67)])
def test_byte_formula_counts_the_mask(h, w, band):
    for n in (1, 7):
        assert split_fetch_bytes(n, h, w, band) == n * int(fetch_mask(h, w, band).sum())


@pytest.mark.parametrize("h,w,labels", [(5, 1, ("Original", "Transformed")), (20, 30, ("Original", "Transformed")),
                                        (135, 241, ("Original", "Transformed")), (64, 96, ("A", "Dog view")),
                                        (300, 161, None), (1080, 1920, ("Original", "HoneyBee"))])
def test_fetching_the_mask_into_the_input_gives_the_split_frame(h, w, labels):
    """Outside the band and the right-hand columns the host split frame IS the input frame."""
    a = np.stack([frames.natural(h, w, 1), frames.noise(h, w, 2)])
    b = np.ascontiguousarray(255 - a[:, ::-1])
    band = 0 if labels is None else tables.split_label_stencil(h, w, *labels).band_rows
    m = fetch_mask(h, w, band).reshape(h, w, 3)
    for seam in (True, False):
        comp = split_compare_batch(torch.from_numpy(a), torch.from_numpy(b), draw_seam=seam).numpy()
        for k in range(len(a)):
            split = draw_split_labels(comp[k].copy(), *labels) if labels is not None else comp[k]
            fetched = a[k].copy()
            fetched[m] = split[m]
            assert np.array_equal(fetched, split), f"{h}x{w} {labels} seam={seam}"


def test_abi_rejects_bad_arguments_before_any_cuda_call():
    from animal_vision_b200 import _abi
    lib = _abi.load()
    n, H, W = 2, 8, 10
    src = np.zeros((n, H, W, 3), np.uint8)
    dst = np.zeros_like(src)
    fs, rs = H * W * 3, W * 3

    def call(s=src.ctypes.data, d=dst.ctypes.data, n=n, H=H, W=W, sfs=fs, srs=rs, dfs=fs, drs=rs, band=3):
        return lib.avb_split_fetch_u8(s, d, n, H, W, sfs, srs, dfs, drs, band, None)
    for kw, msg in ((dict(s=None), b"null"), (dict(d=None), b"null"), (dict(n=0), b"positive"), (dict(n=-1), b"positive"),
                    (dict(H=0), b"positive"), (dict(W=0), b"positive"), (dict(band=H + 1), b"band_rows"),
                    (dict(band=-1), b"band_rows"), (dict(srs=rs - 1), b"row strides"), (dict(drs=rs - 1), b"row strides"),
                    (dict(sfs=-1), b"negative"), (dict(dfs=fs - 1), b"overlap"), (dict(dfs=0), b"overlap"),
                    (dict(dfs=-fs), b"overlap")):
        assert call(**kw) == -1, kw
        assert msg in lib.avb_last_error(), (kw, lib.avb_last_error())
    # well-formed arguments on pageable host memory: refused by the memory check (or a CUDA error without a device)
    assert call() in (-1, -2)
    assert not dst.any()
