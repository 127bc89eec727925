"""JPEG encode on the host (CPU): the header / quantiser builders of animal_vision_b200/tables.py and the NumPy restatement
oracle/jpeg.py are byte-identical to cv2.imencode(".jpg") -- the yardstick of the device encoder (K8)."""
import cv2
import numpy as np
import pytest

import frames
from animal_vision_b200 import tables
from oracle import jpeg as OJ

QUALITIES = (10, 50, 75, 95, 100)
SHAPES = ((1, 1), (7, 9), (8, 8), (16, 16), (17, 33), (37, 53), (135, 241))


def _cv2(img, q):
    ok, enc = cv2.imencode(".jpg", img, [cv2.IMWRITE_JPEG_QUALITY, q])
    assert ok
    return enc.tobytes()


def _segments(data):
    """(marker, payload) of every segment before the entropy-coded data, and the offset where that data starts."""
    out, i = [], 2
    while True:
        m, L = data[i + 1], int.from_bytes(data[i + 2:i + 4], "big")
        out.append((m, data[i + 4:i + 2 + L]))
        i += 2 + L
        if m == 0xDA:
            return out, i


@pytest.mark.parametrize("q", (1, 2, 10, 25, 49, 50, 51, 75, 95, 99, 100))
def test_quant_tables_are_the_dqt_payloads(q):
    segs, _ = _segments(_cv2(frames.natural(37, 53), q))
    dqt = [p for m, p in segs if m == 0xDB]
    qt = tables.jpeg_quant_tables(q)
    assert qt.shape == (2, 64) and qt.dtype == np.uint8
    assert [p[0] for p in dqt] == [0, 1] and [p[1:] for p in dqt] == [qt[0].tobytes(), qt[1].tobytes()]


@pytest.mark.parametrize("q", QUALITIES)
@pytest.mark.parametrize("hw", SHAPES + ((1080, 1920), (65500, 1), (1, 65500)))    # 65500: libjpeg's JPEG_MAX_DIMENSION
def test_header_is_every_byte_before_the_entropy_coded_data(q, hw):
    h, w = hw
    img = frames.constant(h, w, 77) if h * w > 1 << 16 else frames.natural(h, w)
    data = _cv2(img, q)
    _, start = _segments(data)
    assert tables.jpeg_header(h, w, q) == data[:start]


def test_builders_reject_bad_arguments():
    for q in (0, 101, -5):
        with pytest.raises(ValueError):
            tables.jpeg_quant_tables(q)
    for hw in ((0, 5), (5, 0), (65536, 5)):
        with pytest.raises(ValueError):
            tables.jpeg_header(*hw, 95)


@pytest.mark.parametrize("q", QUALITIES)
@pytest.mark.parametrize("hw", SHAPES + ((1080, 1920),))
def test_oracle_is_byte_identical_to_cv2(q, hw):
    for name, img in frames.parity_set(*hw):
        assert OJ.imencode(img, q) == _cv2(img, q), f"{name} {hw} q={q}"
