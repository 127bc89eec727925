"""NumPy restatement of `cv2.imencode(".jpg", bgr_u8, [cv2.IMWRITE_JPEG_QUALITY, q])` with OpenCV's defaults
(libjpeg-turbo: baseline, standard Huffman tables, no restart interval, 4:2:0).

Each stage follows the libjpeg source it restates:
  jcparam.c   jpeg_quality_scaling / jpeg_add_quant_table (baseline: entries clamped to [1, 255])
  jccolor.c   rgb_ycc_convert, 16-bit fixed point
  jcsample.c  h2v2_downsample (bias 1, 2, 1, 2, ...), expand_right_edge
  jcprepct.c  bottom rows replicated to the row group, then each component to a full iMCU row
  jccoefct.c  compress_data: dummy blocks (AC zero, DC copied from the preceding block)
  jcdctmgr.c  level shift, quantisation of the magnitude with round-half-up
  jfdctint.c  jpeg_fdct_islow (CONST_BITS 13, PASS1_BITS 2)
  jchuff.c    DC differences, run/size AC symbols, ZRL, EOB, 0xFF stuffing, 1-padding of the last byte
The entropy coder is vectorised (one symbol per array element) so that 1080p frames encode in about a second."""
from __future__ import annotations

import numpy as np

ZIGZAG = np.array([0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6, 7, 14,
                   21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53,
                   60, 61, 54, 47, 55, 62, 63])

STD_LUMA_Q = np.array([16, 11, 10, 16, 24, 40, 51, 61, 12, 12, 14, 19, 26, 58, 60, 55, 14, 13, 16, 24, 40, 57, 69, 56,
                       14, 17, 22, 29, 51, 87, 80, 62, 18, 22, 37, 56, 68, 109, 103, 77, 24, 35, 55, 64, 81, 104, 113, 92,
                       49, 64, 78, 87, 103, 121, 120, 101, 72, 92, 95, 98, 112, 100, 103, 99])
STD_CHROMA_Q = np.full(64, 99)
STD_CHROMA_Q.reshape(8, 8)[:4, :4] = [[17, 18, 24, 47], [18, 21, 26, 66], [24, 26, 56, 99], [47, 66, 99, 99]]

# ITU-T T.81 Annex K.3: (bits[1..16], values)
DC_LUMA = ([0, 1, 5, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0, 0, 0], list(range(12)))
DC_CHROMA = ([0, 3, 1, 1, 1, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0], list(range(12)))
AC_LUMA = ([0, 2, 1, 3, 3, 2, 4, 3, 5, 5, 4, 4, 0, 0, 1, 0x7d], bytes.fromhex(
    "01020300041105122131410613516107227114328191a1082342b1c11552d1f02433627282090a161718191a25262728292a3435363738"
    "393a434445464748494a535455565758595a636465666768696a737475767778797a838485868788898a92939495969798999aa2a3a4a5"
    "a6a7a8a9aab2b3b4b5b6b7b8b9bac2c3c4c5c6c7c8c9cad2d3d4d5d6d7d8d9dae1e2e3e4e5e6e7e8e9eaf1f2f3f4f5f6f7f8f9fa"))
AC_CHROMA = ([0, 2, 1, 2, 4, 4, 3, 4, 7, 5, 4, 4, 0, 1, 2, 0x77], bytes.fromhex(
    "000102031104052131061241510761711322328108144291a1b1c109233352f0156272d10a162434e125f11718191a262728292a35363738"
    "393a434445464748494a535455565758595a636465666768696a737475767778797a82838485868788898a92939495969798999aa2a3a4a5"
    "a6a7a8a9aab2b3b4b5b6b7b8b9bac2c3c4c5c6c7c8c9cad2d3d4d5d6d7d8d9dae2e3e4e5e6e7e8e9eaf2f3f4f5f6f7f8f9fa"))


def quant_tables(q: int) -> np.ndarray:
    """[2, 64] quantiser values in natural (row-major) order."""
    q = min(max(int(q), 1), 100)
    scale = 5000 // q if q < 50 else 200 - 2 * q
    return np.stack([np.clip((t * scale + 50) // 100, 1, 255) for t in (STD_LUMA_Q, STD_CHROMA_Q)]).astype(np.int64)


def _huff_codes(spec):
    """jchuff.c jpeg_make_c_derived_tbl: symbol -> (code, length)."""
    bits, vals = spec
    code, k, codes, lens = 0, 0, np.zeros(256, np.int64), np.zeros(256, np.int64)
    for L in range(1, 17):
        for _ in range(bits[L - 1]):
            codes[vals[k]], lens[vals[k]] = code, L
            code += 1
            k += 1
        code <<= 1
    return codes, lens


def _segment(marker: int, payload: bytes) -> bytes:
    return bytes([0xFF, marker]) + (len(payload) + 2).to_bytes(2, "big") + payload


def header(H: int, W: int, q: int) -> bytes:
    qt = quant_tables(q)
    out = b"\xff\xd8" + _segment(0xE0, b"JFIF\x00\x01\x01\x00\x00\x01\x00\x01\x00\x00")
    for i in range(2):
        out += _segment(0xDB, bytes([i]) + bytes(qt[i][ZIGZAG].tolist()))
    out += _segment(0xC0, bytes([8]) + H.to_bytes(2, "big") + W.to_bytes(2, "big") + bytes([3, 1, 0x22, 0, 2, 0x11, 1, 3, 0x11, 1]))
    for cls_id, spec in ((0x00, DC_LUMA), (0x10, AC_LUMA), (0x01, DC_CHROMA), (0x11, AC_CHROMA)):
        out += _segment(0xC4, bytes([cls_id]) + bytes(spec[0]) + bytes(spec[1]))
    return out + _segment(0xDA, bytes([3, 1, 0x00, 2, 0x11, 3, 0x11, 0, 63, 0]))


def _fix(x):
    return int(x * 65536 + 0.5)


def rgb_ycc(bgr: np.ndarray):
    """jccolor.c rgb_ycc_convert (input BGR: channel 2 is R)."""
    b, g, r = (bgr[..., i].astype(np.int64) for i in range(3))
    half, off = 1 << 15, 128 << 16
    y = (_fix(0.299) * r + _fix(0.587) * g + _fix(0.114) * b + half) >> 16
    cb = (-_fix(0.16874) * r - _fix(0.33126) * g + _fix(0.5) * b + off + half - 1) >> 16
    cr = (_fix(0.5) * r - _fix(0.41869) * g - _fix(0.08131) * b + off + half - 1) >> 16
    return y, cb, cr


def _descale(x, n):
    return (x + (1 << (n - 1))) >> n


def fdct_islow(blocks: np.ndarray) -> np.ndarray:
    """jfdctint.c on [..., 8, 8] level-shifted int64 samples; output scaled by 8."""
    def pass_(d, last):
        d0, d1, d2, d3, d4, d5, d6, d7 = (d[..., i] for i in range(8))
        tmp0, tmp7, tmp1, tmp6 = d0 + d7, d0 - d7, d1 + d6, d1 - d6
        tmp2, tmp5, tmp3, tmp4 = d2 + d5, d2 - d5, d3 + d4, d3 - d4
        tmp10, tmp13, tmp11, tmp12 = tmp0 + tmp3, tmp0 - tmp3, tmp1 + tmp2, tmp1 - tmp2
        sh = 13 + 2 if last else 13 - 2
        o = [None] * 8
        o[0] = _descale(tmp10 + tmp11, 2) if last else (tmp10 + tmp11) << 2
        o[4] = _descale(tmp10 - tmp11, 2) if last else (tmp10 - tmp11) << 2
        z1 = (tmp12 + tmp13) * 4433
        o[2] = _descale(z1 + tmp13 * 6270, sh)
        o[6] = _descale(z1 - tmp12 * 15137, sh)
        z1, z2, z3, z4 = tmp4 + tmp7, tmp5 + tmp6, tmp4 + tmp6, tmp5 + tmp7
        z5 = (z3 + z4) * 9633
        tmp4, tmp5, tmp6, tmp7 = tmp4 * 2446, tmp5 * 16819, tmp6 * 25172, tmp7 * 12299
        z1, z2, z3, z4 = z1 * -7373, z2 * -20995, z3 * -16069 + z5, z4 * -3196 + z5
        o[7] = _descale(tmp4 + z1 + z3, sh)
        o[5] = _descale(tmp5 + z2 + z4, sh)
        o[3] = _descale(tmp6 + z2 + z3, sh)
        o[1] = _descale(tmp7 + z1 + z4, sh)
        return np.stack(o, -1)
    rows = pass_(blocks.astype(np.int64), False)
    return np.swapaxes(pass_(np.swapaxes(rows, -1, -2), True), -1, -2)


def _blocks(plane: np.ndarray) -> np.ndarray:
    h, w = plane.shape
    return plane.reshape(h // 8, 8, w // 8, 8).transpose(0, 2, 1, 3)


def coefficients(bgr: np.ndarray, q: int):
    """Quantised coefficients in natural order: Y [2*mh, 2*mw, 8, 8], Cb / Cr [mh, mw, 8, 8] per MCU grid (mh x mw),
    dummy blocks included."""
    H, W, _ = bgr.shape
    mh, mw = -(-H // 16), -(-W // 16)
    bh, bw = -(-H // 8), -(-W // 8)                           # luma width_in_blocks / height_in_blocks
    ch, cw = -(-H // 2), -(-W // 2)                           # downsampled chroma size
    y, cb, cr = rgb_ycc(bgr)
    # luma: columns replicated to 8*bw (expand_right_edge), rows to the iMCU row
    yy = np.minimum(np.arange(16 * mh), H - 1)
    xx = np.minimum(np.arange(16 * mw), W - 1)
    Y = y[yy][:, xx]
    # chroma: input columns replicated to 2 * 8 * cwb, rows to the row group (2); h2v2 average; downsampled rows replicated
    cwb = -(-cw // 8)
    cy = np.minimum(np.arange(2 * ch), H - 1)
    cx = np.minimum(np.arange(16 * cwb), W - 1)
    bias = np.tile([1, 2], 4 * cwb)

    def down(p):
        p = p[cy][:, cx]
        s = p[0::2, 0::2] + p[0::2, 1::2] + p[1::2, 0::2] + p[1::2, 1::2]
        return (s + bias) >> 2
    rows_c = np.minimum(np.arange(8 * mh), ch - 1)
    Cb, Cr = down(cb)[rows_c][:, :8 * mw], down(cr)[rows_c][:, :8 * mw]
    qt = quant_tables(q).reshape(2, 8, 8) * 8
    out = []
    for plane, t in ((Y, qt[0]), (Cb, qt[1]), (Cr, qt[1])):
        c = fdct_islow(_blocks(plane) - 128)
        mag = (np.abs(c) + (t >> 1)) // t
        out.append(np.where(c < 0, -mag, mag))
    Yq = out[0]
    # dummy blocks (jccoefct.c compress_data): right edge within an MCU, then the bottom block row of the last MCU row
    if bw % 2:
        Yq[:, bw] = 0
        Yq[:, bw, 0, 0] = Yq[:, bw - 1, 0, 0]
    if bh % 2:
        Yq[bh] = 0
        Yq[bh, 0::2, 0, 0] = Yq[bh - 1, 1::2, 0, 0]
        Yq[bh, 1::2, 0, 0] = Yq[bh - 1, 1::2, 0, 0]
    return Yq, out[1], out[2]


def _nbits(v):
    a = np.abs(v)
    n = np.zeros(a.shape, np.int64)
    nz = a > 0
    n[nz] = np.floor(np.log2(a[nz])).astype(np.int64) + 1
    return n


def entropy(Yq, Cb, Cr) -> bytes:
    mh, mw = Cb.shape[:2]
    y4 = Yq.reshape(mh, 2, mw, 2, 64).transpose(0, 2, 1, 3, 4).reshape(mh * mw, 4, 64)
    blocks = np.concatenate([y4, Cb.reshape(-1, 1, 64), Cr.reshape(-1, 1, 64)], 1)[:, :, ZIGZAG]   # MCU order
    nb = blocks.shape[0] * 6
    comp = np.tile([0, 0, 0, 0, 1, 2], blocks.shape[0])
    coef = blocks.reshape(nb, 64)
    dc = coef[:, 0].copy()
    diff = np.zeros(nb, np.int64)
    for c in range(3):
        idx = np.nonzero(comp == c)[0]
        diff[idx] = np.diff(dc[idx], prepend=0)
    tabs = [_huff_codes(s) for s in (DC_LUMA, AC_LUMA, DC_CHROMA, AC_CHROMA)]
    chroma = (comp > 0).astype(np.int64)
    keys, vals, lens = [], [], []

    def extra(v, n):
        return np.where(v < 0, v - 1, v) & ((1 << n) - 1)

    # DC symbols
    s = _nbits(diff)
    hc = np.where(chroma, tabs[2][0][s], tabs[0][0][s])
    hl = np.where(chroma, tabs[2][1][s], tabs[0][1][s])
    keys.append(np.arange(nb) * 256)
    vals.append((hc << s) | extra(diff, s))
    lens.append(hl + s)
    # AC symbols
    bi, pos = np.nonzero(coef[:, 1:])
    pos = pos + 1
    v = coef[bi, pos]
    prev = np.ones_like(pos)
    first = np.ones(len(bi), bool)
    first[1:] = bi[1:] != bi[:-1]
    prev[~first] = pos[:-1][~first[1:]] + 1
    run = pos - prev
    s = _nbits(v)
    sym = ((run & 15) << 4) | s
    ch = chroma[bi]
    hc = np.where(ch, tabs[3][0][sym], tabs[1][0][sym])
    hl = np.where(ch, tabs[3][1][sym], tabs[1][1][sym])
    keys.append(bi * 256 + 2 * pos + 1)
    vals.append((hc << s) | extra(v, s))
    lens.append(hl + s)
    nzrl = run >> 4                                           # ZRL codes before this coefficient
    rep = np.repeat(np.arange(len(bi)), nzrl)
    keys.append(bi[rep] * 256 + 2 * pos[rep])
    vals.append(np.where(ch[rep], tabs[3][0][0xF0], tabs[1][0][0xF0]))
    lens.append(np.where(ch[rep], tabs[3][1][0xF0], tabs[1][1][0xF0]))
    # EOB where the last AC coefficient is zero
    eob = np.nonzero(coef[:, 63] == 0)[0]
    keys.append(eob * 256 + 255)
    vals.append(np.where(chroma[eob], tabs[3][0][0], tabs[1][0][0]))
    lens.append(np.where(chroma[eob], tabs[3][1][0], tabs[1][1][0]))
    keys, vals, lens = (np.concatenate(a).astype(np.int64) for a in (keys, vals, lens))
    order = np.argsort(keys, kind="stable")
    vals, lens = vals[order], lens[order]
    # MSB-first bit stream, padded with 1-bits to a whole byte
    ev = np.repeat(np.arange(len(lens)), lens)
    start = np.cumsum(lens) - lens
    j = np.arange(len(ev)) - start[ev]
    bits = ((vals[ev] >> (lens[ev] - 1 - j)) & 1).astype(np.uint8)
    pad = (-len(bits)) % 8
    data = np.packbits(np.concatenate([bits, np.ones(pad, np.uint8)]))
    ff = np.nonzero(data == 0xFF)[0]
    return np.insert(data, ff + 1, 0).tobytes()


def imencode(bgr: np.ndarray, quality: int = 95) -> bytes:
    """What cv2.imencode(".jpg", bgr, [cv2.IMWRITE_JPEG_QUALITY, quality]) returns, as bytes."""
    assert bgr.ndim == 3 and bgr.shape[2] == 3 and bgr.dtype == np.uint8
    H, W, _ = bgr.shape
    return header(H, W, quality) + entropy(*coefficients(bgr, quality)) + b"\xff\xd9"
