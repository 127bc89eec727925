"""NumPy restatement of `cv2.imencode(".jpg", bgr_u8, [cv2.IMWRITE_JPEG_QUALITY, q, cv2.IMWRITE_JPEG_OPTIMIZE, 1])`: the
file of oracle/jpeg.py (OpenCV's defaults: libjpeg-turbo baseline, 4:2:0, no restart interval) with Huffman tables built
from the frame's own symbol counts (jchuff.c htest_one_block / jpeg_gen_optimal_table) -- the yardstick of K8's optimized
mode.  The file differs from the standard one only in the payloads of the four DHT segments and in the codes of the
entropy-coded data (same DC prediction, ZRL, EOB, stuffing and padding).  The coefficients, the standard header and the
Huffman code derivation are oracle/jpeg.py's; the symbol and bit-stream stages are restated here with the tables as an
argument."""
from __future__ import annotations

import numpy as np

from oracle.jpeg import (AC_CHROMA, AC_LUMA, DC_CHROMA, DC_LUMA, ZIGZAG, _huff_codes, _nbits, _segment, coefficients,
                         header)
from oracle.jpeg import imencode as oracle_imencode


def _symbols(Yq, Cb, Cr):
    """Every block in MCU order (Y00 Y01 Y10 Y11 Cb Cr) and the symbols the coder emits for it: (coef [nb, 64] zigzag,
    chroma flag per block, DC difference per block, and per nonzero AC coefficient its block, zigzag position, value and
    the zero run before it)."""
    mh, mw = Cb.shape[:2]
    y4 = Yq.reshape(mh, 2, mw, 2, 64).transpose(0, 2, 1, 3, 4).reshape(mh * mw, 4, 64)
    coef = np.concatenate([y4, Cb.reshape(-1, 1, 64), Cr.reshape(-1, 1, 64)], 1)[:, :, ZIGZAG].reshape(-1, 64)
    comp = np.tile([0, 0, 0, 0, 1, 2], coef.shape[0] // 6)
    diff = np.zeros(len(coef), np.int64)
    for c in range(3):
        idx = np.nonzero(comp == c)[0]
        diff[idx] = np.diff(coef[idx, 0], prepend=0)
    bi, pos = np.nonzero(coef[:, 1:])
    pos = pos + 1
    prev = np.ones_like(pos)
    first = np.ones(len(bi), bool)
    first[1:] = bi[1:] != bi[:-1]
    prev[~first] = pos[:-1][~first[1:]] + 1
    return coef, (comp > 0).astype(np.int64), diff, bi, pos, coef[bi, pos], pos - prev


def statistics(Yq, Cb, Cr) -> np.ndarray:
    """[4, 256] int64 counts of the symbols the coder emits (jchuff.c htest_one_block), tables DC0, AC0, DC1, AC1: one
    DC size per block, (run << 4) | size per nonzero AC coefficient, 0xF0 per 16 zeros before one, and an EOB (0x00)
    for each block that ends in zeros.  Dummy blocks count like any other."""
    coef, chroma, diff, bi, pos, v, run = _symbols(Yq, Cb, Cr)
    freq = np.zeros((4, 256), np.int64)
    np.add.at(freq, (2 * chroma, _nbits(diff)), 1)
    ch = chroma[bi]
    np.add.at(freq, (2 * ch + 1, ((run & 15) << 4) | _nbits(v)), 1)
    np.add.at(freq, (2 * ch + 1, 0xF0), run >> 4)
    np.add.at(freq, (2 * chroma[coef[:, 63] == 0] + 1, 0), 1)
    return freq


def gen_optimal_table(freq):
    """jchuff.c jpeg_gen_optimal_table: 256 symbol counts -> ((bits[1..16], values), whether a code longer than 16 bits
    had to be shortened)."""
    freq = [int(x) for x in freq] + [1]                     # symbol 256: reserves the all-ones code point
    codesize, others = [0] * 257, [-1] * 257
    while True:
        c1 = c2 = -1
        v = 1000000000
        for i in range(257):                                # the smallest count, ties to the largest symbol
            if freq[i] and freq[i] <= v:
                v, c1 = freq[i], i
        v = 1000000000
        for i in range(257):
            if freq[i] and freq[i] <= v and i != c1:
                v, c2 = freq[i], i
        if c2 < 0:
            break
        freq[c1] += freq[c2]
        freq[c2] = 0
        codesize[c1] += 1
        while others[c1] >= 0:
            c1 = others[c1]
            codesize[c1] += 1
        others[c1] = c2
        codesize[c2] += 1
        while others[c2] >= 0:
            c2 = others[c2]
            codesize[c2] += 1
    bits = [0] * 33
    for c in codesize:
        if c:
            bits[c] += 1
    limited = any(bits[17:])
    for i in range(32, 16, -1):
        while bits[i] > 0:
            j = i - 2
            while bits[j] == 0:
                j -= 1
            bits[i] -= 2
            bits[i - 1] += 1
            bits[j + 1] += 2
            bits[j] -= 1
    i = 16
    while bits[i] == 0:
        i -= 1
    bits[i] -= 1
    vals = [s for L in range(1, 33) for s in range(256) if codesize[s] == L]
    return (bits[1:17], vals), limited


def optimal_tables(Yq, Cb, Cr):
    """The (bits, values) of the DC0, AC0, DC1 and AC1 tables libjpeg builds for these coefficients, and whether any of
    them had codes shortened to 16 bits."""
    built = [gen_optimal_table(f) for f in statistics(Yq, Cb, Cr)]
    return tuple(t for t, _ in built), any(lim for _, lim in built)


def header_with(H: int, W: int, q: int, huff) -> bytes:
    """`header` with the DHT payloads of `huff`, the (bits, values) of DC0, AC0, DC1, AC1."""
    std = header(H, W, q)
    dht = b"".join(_segment(0xC4, bytes([c]) + bytes(b) + bytes(v)) for c, (b, v) in zip((0x00, 0x10, 0x01, 0x11), huff))
    sos = 14                                                # the SOS segment closes the header
    pre = len(std) - sos - sum(4 + 1 + 16 + len(v) for _, v in (DC_LUMA, AC_LUMA, DC_CHROMA, AC_CHROMA))
    return std[:pre] + dht + std[-sos:]


def entropy_with(Yq, Cb, Cr, huff) -> bytes:
    """`entropy` with the codes of `huff`."""
    coef, chroma, diff, bi, pos, v, run = _symbols(Yq, Cb, Cr)
    nb = len(coef)
    tabs = [_huff_codes(s) for s in huff]

    def extra(v, n):
        return np.where(v < 0, v - 1, v) & ((1 << n) - 1)

    def code(t, sym):                                       # t: table 0 (DC) or 1 (AC); codes and lengths per element
        ch = chroma if t == 0 else chroma[bi]
        return (np.where(ch, tabs[t + 2][0][sym], tabs[t][0][sym]), np.where(ch, tabs[t + 2][1][sym], tabs[t][1][sym]))

    s = _nbits(diff)
    hc, hl = code(0, s)
    keys, vals, lens = [np.arange(nb) * 256], [(hc << s) | extra(diff, s)], [hl + s]
    s = _nbits(v)
    hc, hl = code(1, ((run & 15) << 4) | s)
    keys.append(bi * 256 + 2 * pos + 1)
    vals.append((hc << s) | extra(v, s))
    lens.append(hl + s)
    rep = np.repeat(np.arange(len(bi)), run >> 4)            # ZRL codes before this coefficient
    zc, zl = (np.where(chroma[bi[rep]], tabs[3][k][0xF0], tabs[1][k][0xF0]) for k in (0, 1))
    keys.append(bi[rep] * 256 + 2 * pos[rep])
    vals.append(zc)
    lens.append(zl)
    eob = np.nonzero(coef[:, 63] == 0)[0]
    keys.append(eob * 256 + 255)
    vals.append(np.where(chroma[eob], tabs[3][0][0], tabs[1][0][0]))
    lens.append(np.where(chroma[eob], tabs[3][1][0], tabs[1][1][0]))
    keys, vals, lens = (np.concatenate(a).astype(np.int64) for a in (keys, vals, lens))
    order = np.argsort(keys, kind="stable")
    vals, lens = vals[order], lens[order]
    ev = np.repeat(np.arange(len(lens)), lens)
    j = np.arange(len(ev)) - (np.cumsum(lens) - lens)[ev]
    bits = ((vals[ev] >> (lens[ev] - 1 - j)) & 1).astype(np.uint8)
    data = np.packbits(np.concatenate([bits, np.ones((-len(bits)) % 8, np.uint8)]))
    return np.insert(data, np.nonzero(data == 0xFF)[0] + 1, 0).tobytes()


def imencode(bgr: np.ndarray, quality: int = 95, optimize: bool = False) -> bytes:
    """What cv2.imencode(".jpg", bgr, [cv2.IMWRITE_JPEG_QUALITY, quality]) returns, as bytes (oracle.jpeg.imencode); with
    `optimize`, what it returns with cv2.IMWRITE_JPEG_OPTIMIZE set as well."""
    if not optimize:
        return oracle_imencode(bgr, quality)
    assert bgr.ndim == 3 and bgr.shape[2] == 3 and bgr.dtype == np.uint8
    H, W, _ = bgr.shape
    co = coefficients(bgr, quality)
    huff = optimal_tables(*co)[0]
    return header_with(H, W, quality, huff) + entropy_with(*co, huff) + b"\xff\xd9"
