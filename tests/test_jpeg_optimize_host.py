"""Optimized Huffman tables on the host (CPU): the NumPy restatement tests/jpeg_optimize_oracle.py
`imencode(..., optimize=True)` is byte-identical to cv2.imencode(".jpg") with IMWRITE_JPEG_OPTIMIZE -- the yardstick of
K8's optimized mode -- and the header pieces of animal_vision_b200/tables.py that mode takes rebuild the standard header."""
import cv2
import numpy as np
import pytest

import frames
import jpeg_optimize_oracle as OJ
from animal_vision_b200 import tables

QUALITIES = (1, 10, 50, 75, 95, 100)
SHAPES = ((1, 1), (7, 9), (8, 8), (16, 16), (17, 33), (37, 53), (135, 241))


def _cv2_opt(img, q):
    ok, enc = cv2.imencode(".jpg", img, [cv2.IMWRITE_JPEG_QUALITY, q, cv2.IMWRITE_JPEG_OPTIMIZE, 1])
    assert ok
    return enc.tobytes()


@pytest.mark.parametrize("q", QUALITIES)
@pytest.mark.parametrize("hw", SHAPES)
def test_oracle_optimized_equals_cv2(q, hw):
    for name, img in frames.parity_set(*hw):
        assert OJ.imencode(img, q, optimize=True) == _cv2_opt(img, q), f"{name} {hw} q={q}"


def test_code_length_limiting_branch():
    """A 720p natural frame at q100 has symbols rare enough for codes longer than 16 bits: the branch that folds them
    down runs, and the file still equals cv2's."""
    img = frames.natural(720, 1280, 4)
    _, limited = OJ.optimal_tables(*OJ.coefficients(img, 100))
    assert limited
    assert OJ.imencode(img, 100, optimize=True) == _cv2_opt(img, 100)


@pytest.mark.parametrize("q", (75, 95))
def test_constant_frame_has_one_symbol_per_table(q):
    img = frames.constant(48, 64, 128)                     # Y = Cb = Cr = 128: every DC difference is 0
    (dc0, ac0, dc1, ac1), limited = OJ.optimal_tables(*OJ.coefficients(img, q))
    assert not limited
    for bits, vals in (dc0, ac0, dc1, ac1):
        assert len(vals) == 1 and sum(bits) == 1
    assert dc0[1] == dc1[1] == ac0[1] == ac1[1] == [0]     # DC size 0, EOB
    assert OJ.imencode(img, q, optimize=True) == _cv2_opt(img, q)


def test_rgb_input_through_a_channel_swap():
    rgb = frames.natural(37, 53, 2)
    assert OJ.imencode(np.ascontiguousarray(rgb[..., ::-1]), 90, optimize=True) == _cv2_opt(rgb[..., ::-1], 90)


def test_optimized_file_differs_only_in_the_dht_payloads_and_the_data():
    img = frames.natural(135, 241)
    std, opt = OJ.imencode(img, 75), OJ.imencode(img, 75, optimize=True)
    assert len(opt) < len(std)
    pre = tables.jpeg_header_prefix(135, 241, 75)
    assert std.startswith(pre) and opt.startswith(pre)
    assert std[len(pre):len(pre) + 2] == opt[len(pre):len(pre) + 2] == b"\xff\xc4"
    assert tables.JPEG_SOS in opt


@pytest.mark.parametrize("q", (1, 50, 95, 100))
@pytest.mark.parametrize("hw", ((1, 1), (37, 53), (1080, 1920)))
def test_header_pieces_with_the_standard_tables_are_the_header(q, hw):
    std = OJ.header(*hw, q)
    dht = b"".join(OJ._segment(0xC4, bytes([c]) + bytes(b) + bytes(v))
                   for c, (b, v) in zip((0x00, 0x10, 0x01, 0x11), (OJ.DC_LUMA, OJ.AC_LUMA, OJ.DC_CHROMA, OJ.AC_CHROMA)))
    assert tables.jpeg_header_prefix(*hw, q) + dht + tables.JPEG_SOS == tables.jpeg_header(*hw, q) == std
    assert OJ.header_with(*hw, q, (OJ.DC_LUMA, OJ.AC_LUMA, OJ.DC_CHROMA, OJ.AC_CHROMA)) == std


def test_header_prefix_rejects_bad_arguments():
    for hw in ((0, 5), (5, 0), (65536, 5)):
        with pytest.raises(ValueError):
            tables.jpeg_header_prefix(*hw, 95)
    with pytest.raises(ValueError):
        tables.jpeg_header_prefix(8, 8, 0)


def test_host_route_of_the_server_sets_the_flag():
    """FrameBatcher's host encode ("human" requests, NumPy runners) passes IMWRITE_JPEG_OPTIMIZE for optimized requests."""
    from animal_vision_b200.serving import FrameBatcher, _split_host
    img = frames.natural(64, 96, 3)
    view = np.ascontiguousarray(img[..., ::-1])
    with FrameBatcher(run_batch=lambda key, b: b[..., ::-1].copy()) as fb:
        std = fb.submit_jpeg(img, "human").result(10)
        opt = fb.submit_jpeg(img, "human", optimize=True).result(10)
        ran = fb.submit_jpeg(img, "dog", optimize=True).result(10)
        split = fb.submit_split_jpeg(img, "dog", optimize=True).result(10)
    assert std == cv2.imencode(".jpg", img)[1].tobytes()
    assert opt == _cv2_opt(img, 95) and len(opt) < len(std)
    assert ran == _cv2_opt(view, 95)
    assert split == _split_host(img, view, ("Original", "Transformed"), True, True)
    assert split != _split_host(img, view, ("Original", "Transformed"), True)
