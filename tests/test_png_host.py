"""PNG encode on the host (CPU): the header builder of animal_vision_b200/tables.py and the NumPy restatement
oracle/png.py are byte-identical to cv2.imencode(".png") -- the yardstick of the device encoder (K10) -- and the
oracle's deflate equals Python's zlib with the same settings (level 1, Z_RLE, memLevel 8) on arbitrary bytes."""
import struct
import zlib

import cv2
import numpy as np
import pytest

import frames
from animal_vision_b200 import tables
from oracle import png as OP

# W == 1, H == 1, and filtered sizes either side of libpng's 16384-byte window rewrite (H * (3W + 1))
SHAPES = ((1, 1), (1, 2), (2, 1), (3, 7), (5, 5), (17, 33), (40, 41), (61, 89), (300, 1), (1, 5000), (1, 5461), (1, 5462),
          (128, 42), (129, 42), (130, 42), (135, 241))


def _cv2(img):
    ok, enc = cv2.imencode(".png", img)
    assert ok
    return enc.tobytes()


def _chunks(data):
    out, i = [], 8
    while i < len(data):
        n = struct.unpack(">I", data[i:i + 4])[0]
        out.append((data[i + 4:i + 8], n))
        i += 12 + n
    return out


@pytest.mark.parametrize("hw", SHAPES + ((1080, 1920),))
def test_oracle_is_byte_identical_to_cv2(hw):
    for name, img in frames.parity_set(*hw):
        assert OP.imencode(img) == _cv2(img), f"{name} {hw}"


def _stored_block_lengths(d: bytes):
    """LEN of every leading stored block of a raw deflate stream, and whether the stream ended on one of them."""
    lens, bit = [], 0
    while True:
        hdr = (d[bit >> 3] | (d[(bit >> 3) + 1] << 8) if (bit >> 3) + 1 < len(d) else d[bit >> 3]) >> (bit & 7)
        final, btype = hdr & 1, (hdr >> 1) & 3
        if btype != 0:
            return lens, False
        i = ((bit + 3) + 7) >> 3
        n, nn = struct.unpack("<HH", d[i:i + 4])
        assert n ^ nn == 0xFFFF
        lens.append(n)
        bit = 8 * (i + 4 + n)
        if final:
            return lens, bit == 8 * len(d)


def test_noise_codes_as_stored_blocks_past_the_window():
    """Noise is all literals, so every block is stored, 16383 bytes each: the window argument of DESIGN.md K10 on a
    stream (389 070 bytes) several times zlib's 64 KB window."""
    img = frames.noise(270, 480, 7)
    f = OP.filtered(img)
    assert f.size > 4 * 65536
    d = OP.deflate(f)
    lens, ended = _stored_block_lengths(d)
    assert ended and sum(lens) == f.size
    assert lens[:-1] == [OP.BLOCK_SYMBOLS] * (len(lens) - 1) and 0 < lens[-1] <= OP.BLOCK_SYMBOLS
    assert zlib.decompress(b"".join(_idat_payloads(_cv2(img)))) == f.tobytes()
    assert OP.imencode(img) == _cv2(img)


def _idat_payloads(data):
    out, i = [], 8
    while i < len(data):
        n = struct.unpack(">I", data[i:i + 4])[0]
        if data[i + 4:i + 8] == b"IDAT":
            out.append(data[i + 8:i + 8 + n])
        i += 12 + n
    return out


@pytest.mark.parametrize("v", (0, 77, 255))
def test_flat_frames_code_as_258_byte_matches(v):
    img = frames.constant(720, 1280, v)
    sym, _ = OP.parse(OP.filtered(img))
    assert (sym == 256 + 258 - 3).sum() > 1000
    assert OP.imencode(img) == _cv2(img)


@pytest.mark.parametrize("hw", ((129, 42), (258, 42), (6, 1820)))
def test_symbol_count_multiple_of_block_size(hw):
    """A symbol count that is a multiple of 16383 ends in zlib's empty final block (Z_FINISH)."""
    img = frames.noise(*hw, 0)
    sym, _ = OP.parse(OP.filtered(img))
    assert sym.size % OP.BLOCK_SYMBOLS == 0
    assert OP.imencode(img) == _cv2(img)


@pytest.mark.parametrize("hw", ((5, 1637), (20, 409), (80, 102)))
def test_zlib_stream_of_whole_idat_payloads(hw):
    """A zlib stream of exactly 3 * 8192 bytes: libpng writes three full IDAT chunks and no empty one."""
    img = frames.noise(*hw, 1)
    data = _cv2(img)
    assert [c for c in _chunks(data)] == [(b"IHDR", 13), (b"IDAT", 8192), (b"IDAT", 8192), (b"IDAT", 8192), (b"IEND", 0)]
    assert OP.imencode(img) == data


def _run_bytes(rng, n):
    vals = rng.integers(0, 256, int(rng.integers(1, 40)), dtype=np.uint8)
    lens = rng.geometric(1 / float(rng.choice([1.2, 2.5, 8, 60, 400])), size=n)
    return np.repeat(rng.choice(vals, size=n), lens).astype(np.uint8)


def _zlib_rle(b: bytes) -> bytes:
    co = zlib.compressobj(1, zlib.DEFLATED, 15, 8, zlib.Z_RLE)
    return co.compress(b) + co.flush()


@pytest.mark.parametrize("seed", range(24))
def test_deflate_equals_zlib_rle_on_run_structured_bytes(seed):
    rng = np.random.default_rng(seed)
    s = _run_bytes(rng, int(rng.integers(1, 60000)))
    z = _zlib_rle(s.tobytes())
    assert OP.deflate(s) == z[2:-4]
    assert struct.pack(">I", OP.adler32(s)) == z[-4:]


def test_deflate_equals_zlib_on_skewed_histograms():
    """Fibonacci-like symbol counts push Huffman depths past 15 (gen_bitlen's overflow fix)."""
    fib = [1, 1]
    while len(fib) < 22:
        fib.append(fib[-1] + fib[-2])
    rng = np.random.default_rng(11)
    for total in (16000, 40000):
        counts = np.array(fib[:22], np.int64)
        counts = np.maximum(1, counts * total // counts.sum())
        s = np.repeat(np.arange(0, 2 * len(counts), 2, dtype=np.uint8), counts)
        rng.shuffle(s)
        assert OP.deflate(s) == _zlib_rle(s.tobytes())[2:-4]


def test_deflate_edge_lengths():
    for n in (1, 2, 3, 4, 5, 258, 259, 260, 261, 262, 517, 518, 16383, 16384, 32766):
        for s in (np.zeros(n, np.uint8), np.arange(n, dtype=np.uint8), np.repeat(np.arange(n, dtype=np.uint8), 4)[:n]):
            assert OP.deflate(s) == _zlib_rle(s.tobytes())[2:-4], n


@pytest.mark.parametrize("hw", ((1, 1), (1, 5461), (1, 5462), (3, 3), (8, 8), (17, 33), (54, 100), (1080, 1920),
                                (65535, 1), (1, 65535)))
def test_header_is_signature_ihdr_and_zlib_header(hw):
    h, w = hw
    img = frames.constant(h, w, 9) if h * w > 1 << 16 else frames.natural(h, w)
    data = _cv2(img)
    assert tables.png_header(h, w) == OP.header(h, w) == data[:33] + data[41:43]


def test_header_rejects_bad_sizes():
    for hw in ((0, 5), (5, 0), (65536, 5), (5, 65536)):
        with pytest.raises(ValueError):
            tables.png_header(*hw)
