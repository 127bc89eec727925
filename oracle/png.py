"""NumPy restatement of `cv2.imencode(".png", bgr_u8)` with OpenCV's defaults (libpng 1.6, zlib 1.2.11: compression
level 1, strategy Z_RLE, memLevel 8, filter Sub).

Each stage follows the source it restates:
  pngwutil.c  signature, IHDR (depth 8, colour type 2, no interlace), IDAT payloads of 8192 bytes (the zbuffer size),
              IEND; optimize_cmf: CMF / FLG rewritten to the smallest window that holds <= 16384 bytes of image data
  png.c / pngwutil.c  png_write_filtered_row with filter Sub only: f[i] = x[i] - x[i-3] mod 256, first pixel copied,
              RGB byte order (cv2 swaps BGR); a one-pixel-wide row takes filter None
  deflate.c   deflate_rle: a match (distance 1) only where f[p-1] == f[p] == f[p+1] == f[p+2], extended while bytes
              equal f[p-1], up to 258.  So each maximal run of R equal bytes codes as one literal, (R-1) // 258 matches
              of 258, then the rest r = (R-1) % 258 as one match if r >= 3, else r literals; no match crosses a change
              of byte value.  _tr_tally: a block is flushed after every 16383 symbols (lit_bufsize - 1, memLevel 8),
              and Z_FINISH flushes a final block with whatever is left, possibly nothing.
  trees.c     _tr_flush_block: build_tree (heap order, depth tie-break, gen_bitlen overflow fix), build_bl_tree /
              scan_tree / send_tree, opt_len against static_len against stored_len + 4; _tr_stored_block
  adler32.c   Adler-32 of the filtered bytes, big-endian after the deflate data
The bit packer is vectorised; only the per-block tree construction is a Python loop."""
from __future__ import annotations

import struct
import zlib as _zlib_crc   # crc32 only: the chunk CRC is not what is being restated here

import numpy as np

SIGNATURE = b"\x89PNG\r\n\x1a\n"
IDAT_PAYLOAD = 8192                 # libpng's zbuffer size: every IDAT but the last carries exactly this much
BLOCK_SYMBOLS = 16383               # lit_bufsize - 1 with memLevel 8
MAX_MATCH = 258

L_CODES, D_CODES, BL_CODES = 286, 30, 19
END_BLOCK = 256
EXTRA_LBITS = [0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0]
EXTRA_DBITS = [0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13]
EXTRA_BLBITS = [0] * 16 + [2, 3, 7]
BL_ORDER = [16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15]


def _length_tables():
    """trees.c tr_static_init: base_length[code] and _length_code[len - 3]."""
    base, code_of = [0] * 29, [0] * 256
    length = 0
    for code in range(28):
        base[code] = length
        for _ in range(1 << EXTRA_LBITS[code]):
            code_of[length] = code
            length += 1
    code_of[length - 1] = 28          # length 258 goes to code 285, overwriting 284's last slot
    return np.array(base, np.int64), np.array(code_of, np.int64)


BASE_LENGTH, LENGTH_CODE = _length_tables()


def _bi_reverse(code, n):
    r = 0
    for _ in range(n):
        r = (r << 1) | (code & 1)
        code >>= 1
    return r


def _gen_codes(lens, max_code, bl_count):
    next_code, code = [0] * 16, 0
    for bits in range(1, 16):
        code = (code + bl_count[bits - 1]) << 1
        next_code[bits] = code
    codes = [0] * len(lens)
    for n in range(max_code + 1):
        ln = lens[n]
        if ln:
            codes[n] = _bi_reverse(next_code[ln], ln)
            next_code[ln] += 1
    return codes


def _static_trees():
    lens = [8] * 144 + [9] * 112 + [7] * 24 + [8] * 8
    bl_count = [0] * 16
    for ln in lens:
        bl_count[ln] += 1
    lcodes = _gen_codes(lens, 287, bl_count)
    return lens, lcodes, [5] * D_CODES, [_bi_reverse(n, 5) for n in range(D_CODES)]


STATIC_LLEN, STATIC_LCODE, STATIC_DLEN, STATIC_DCODE = _static_trees()


class _Tree:
    """One trees.c tree_desc after build_tree: Len / Code per symbol and max_code."""

    def __init__(self, freq, elems, max_length, extra, base, stree_len):
        self.freq = list(freq) + [0] * (2 * elems + 1 - len(freq))
        self.elems, self.max_length, self.extra, self.base, self.stree_len = elems, max_length, extra, base, stree_len


def build_tree(state, t: _Tree):
    """trees.c build_tree + gen_bitlen + gen_codes.  state: dict with opt_len / static_len (updated in place)."""
    elems, freq = t.elems, t.freq
    HEAP_SIZE = 2 * L_CODES + 1
    heap = [0] * HEAP_SIZE
    depth = [0] * (2 * L_CODES + 1)
    dad = [0] * (2 * elems + 1)
    length = [0] * (2 * elems + 1)
    heap_len, heap_max, max_code = 0, HEAP_SIZE, -1
    for n in range(elems):
        if freq[n]:
            heap_len += 1
            heap[heap_len] = max_code = n
            depth[n] = 0
    while heap_len < 2:
        heap_len += 1
        if max_code < 2:
            max_code += 1
            node = max_code
        else:
            node = 0
        heap[heap_len] = node
        freq[node] = 1
        depth[node] = 0
        state["opt_len"] -= 1
        if t.stree_len is not None:
            state["static_len"] -= t.stree_len[node]

    def smaller(n, m):
        return freq[n] < freq[m] or (freq[n] == freq[m] and depth[n] <= depth[m])

    def downheap(k):
        v = heap[k]
        j = k << 1
        while j <= heap_len:
            if j < heap_len and smaller(heap[j + 1], heap[j]):
                j += 1
            if smaller(v, heap[j]):
                break
            heap[k] = heap[j]
            k = j
            j <<= 1
        heap[k] = v

    for n in range(heap_len // 2, 0, -1):
        downheap(n)
    node = elems
    while True:
        n = heap[1]                                   # pqremove
        heap[1] = heap[heap_len]
        heap_len -= 1
        downheap(1)
        m = heap[1]
        heap_max -= 1
        heap[heap_max] = n
        heap_max -= 1
        heap[heap_max] = m
        freq[node] = freq[n] + freq[m]
        depth[node] = max(depth[n], depth[m]) + 1
        dad[n] = dad[m] = node
        heap[1] = node
        node += 1
        downheap(1)
        if heap_len < 2:
            break
    heap_max -= 1
    heap[heap_max] = heap[1]

    # gen_bitlen
    bl_count = [0] * 16
    length[heap[heap_max]] = 0
    overflow = 0
    h = heap_max + 1
    while h < HEAP_SIZE:
        n = heap[h]
        bits = length[dad[n]] + 1
        if bits > t.max_length:
            bits, overflow = t.max_length, overflow + 1
        length[n] = bits
        h += 1
        if n > max_code:
            continue
        bl_count[bits] += 1
        xbits = t.extra[n - t.base] if n >= t.base else 0
        f = freq[n]
        state["opt_len"] += f * (bits + xbits)
        if t.stree_len is not None:
            state["static_len"] += f * (t.stree_len[n] + xbits)
    if overflow:
        while True:
            bits = t.max_length - 1
            while bl_count[bits] == 0:
                bits -= 1
            bl_count[bits] -= 1
            bl_count[bits + 1] += 2
            bl_count[t.max_length] -= 1
            overflow -= 2
            if overflow <= 0:
                break
        h = HEAP_SIZE
        for bits in range(t.max_length, 0, -1):
            n = bl_count[bits]
            while n != 0:
                h -= 1
                m = heap[h]
                if m > max_code:
                    continue
                if length[m] != bits:
                    state["opt_len"] += (bits - length[m]) * freq[m]
                    length[m] = bits
                n -= 1
    lens = length[:elems]
    t.lens, t.max_code = lens, max_code
    t.codes = _gen_codes(lens, max_code, bl_count)
    return t


def _tree_runs(lens, max_code):
    """scan_tree / send_tree: the code-length alphabet symbols (sym, extra value, extra bits) describing lens[0..max_code]."""
    out = []
    prevlen, nextlen, count = -1, lens[0], 0
    max_count, min_count = (138, 3) if nextlen == 0 else (7, 4)
    ext = list(lens[:max_code + 1]) + [0xFFFF]        # the guard
    for n in range(max_code + 1):
        curlen, nextlen = nextlen, ext[n + 1]
        count += 1
        if count < max_count and curlen == nextlen:
            continue
        if count < min_count:
            out += [(curlen, 0, 0)] * count
        elif curlen != 0:
            if curlen != prevlen:
                out.append((curlen, 0, 0))
                count -= 1
            out.append((16, count - 3, 2))
        elif count <= 10:
            out.append((17, count - 3, 3))
        else:
            out.append((18, count - 11, 7))
        count, prevlen = 0, curlen
        if nextlen == 0:
            max_count, min_count = 138, 3
        elif curlen == nextlen:
            max_count, min_count = 6, 3
        else:
            max_count, min_count = 7, 4
    return out


def block_plan(lit_freq, n_matches, stored_len):
    """_tr_flush_block's choice for one block.  lit_freq: length-286 symbol counts (END_BLOCK included); n_matches:
    count of distance code 0.  Returns (kind, llen, lcode, dlen, dcode, header) with kind 0 stored, 1 static,
    2 dynamic, and header the (value, bits) list of a dynamic block's tree description."""
    state = {"opt_len": 0, "static_len": 0}
    lt = build_tree(state, _Tree(lit_freq, L_CODES, 15, EXTRA_LBITS, 257, STATIC_LLEN))
    dt = build_tree(state, _Tree([n_matches] + [0] * (D_CODES - 1), D_CODES, 15, EXTRA_DBITS, 0, STATIC_DLEN))
    runs = _tree_runs(lt.lens, lt.max_code) + _tree_runs(dt.lens, dt.max_code)
    blfreq = [0] * BL_CODES
    for s, _, _ in runs:
        blfreq[s] += 1
    bt = build_tree(state, _Tree(blfreq, BL_CODES, 7, EXTRA_BLBITS, 0, None))
    max_blindex = BL_CODES - 1
    while max_blindex >= 3 and bt.lens[BL_ORDER[max_blindex]] == 0:
        max_blindex -= 1
    state["opt_len"] += 3 * (max_blindex + 1) + 5 + 5 + 4
    opt_lenb = (state["opt_len"] + 3 + 7) >> 3
    static_lenb = (state["static_len"] + 3 + 7) >> 3
    if static_lenb <= opt_lenb:
        opt_lenb = static_lenb
    if stored_len + 4 <= opt_lenb:
        return 0, None, None, None, None, None
    if static_lenb == opt_lenb:
        return 1, STATIC_LLEN, STATIC_LCODE, STATIC_DLEN, STATIC_DCODE, None
    header = [(lt.max_code + 1 - 257, 5), (dt.max_code + 1 - 1, 5), (max_blindex + 1 - 4, 4)]
    header += [(bt.lens[BL_ORDER[r]], 3) for r in range(max_blindex + 1)]
    for s, v, nb in runs:
        header.append((bt.codes[s], bt.lens[s]))
        if nb:
            header.append((v, nb))
    return 2, lt.lens, lt.codes, dt.lens, dt.codes, header


def filtered(bgr: np.ndarray) -> np.ndarray:
    """The filtered image data: per row a filter-type byte (1 Sub, or 0 None for W == 1), then the filtered RGB bytes."""
    H, W, _ = bgr.shape
    x = np.ascontiguousarray(bgr[:, :, ::-1]).reshape(H, 3 * W)
    f = x.copy()
    f[:, 3:] = x[:, 3:] - x[:, :-3]                   # uint8 wraps mod 256
    ftype = np.full((H, 1), 1 if W > 1 else 0, np.uint8)
    return np.concatenate([ftype, f], 1).reshape(-1)


def parse(f: np.ndarray):
    """deflate_rle's symbols in closed form.  Returns (sym, pos): sym < 256 a literal byte, 256 + (len - 3) a match of
    distance 1; pos the first filtered byte each symbol covers."""
    S = f.size
    starts = np.concatenate([[0], np.nonzero(f[1:] != f[:-1])[0] + 1]).astype(np.int64)
    R = np.diff(np.concatenate([starts, [S]]))
    m, r = (R - 1) // MAX_MATCH, (R - 1) % MAX_MATCH
    tail = np.where(r >= 3, 1, r)
    cnt = 1 + m + tail
    run = np.repeat(np.arange(starts.size), cnt)
    j = np.arange(run.size) - np.repeat(np.cumsum(cnt) - cnt, cnt)
    s, mm, rr = starts[run], m[run], r[run]
    rest = s + 1 + MAX_MATCH * mm
    pos = np.where(j == 0, s, np.where(j <= mm, s + 1 + MAX_MATCH * (j - 1), rest + np.where(rr >= 3, 0, j - mm - 1)))
    is_match = (j > 0) & ((j <= mm) | (rr >= 3))
    mlen = np.where(j <= mm, MAX_MATCH, rr)
    sym = np.where(is_match, 256 + mlen - 3, f[s].astype(np.int64))
    return sym, pos


def _pack(vals, lens, bitpos):
    """LSB-first bit packing of (value, length) pairs starting at bit offset bitpos (< 8); returns (bytes array, end bit
    offset relative to the first byte)."""
    vals = np.asarray(vals, np.int64)
    lens = np.asarray(lens, np.int64)
    end = np.cumsum(lens) + bitpos
    start = end - lens
    nbytes = (int(end[-1]) + 7) >> 3 if lens.size else 0
    out = np.zeros(nbytes + 4, np.float64)
    bi, sh = start >> 3, start & 7
    v = vals << sh                                    # <= 20 + 7 bits
    for k in range(4):
        out += np.bincount(bi + k, weights=((v >> (8 * k)) & 255).astype(np.float64), minlength=nbytes + 4)[:nbytes + 4]
    return out[:nbytes].astype(np.uint8), int(end[-1]) if lens.size else bitpos


def deflate(f: np.ndarray) -> bytes:
    """The raw deflate stream zlib.compressobj(1, DEFLATED, wbits, 8, Z_RLE) writes for f (no zlib header/trailer)."""
    sym, pos = parse(f)
    T, S = sym.size, f.size
    nblocks = T // BLOCK_SYMBOLS + 1
    bstart = np.append(pos[::BLOCK_SYMBOLS][:nblocks], [S] * (nblocks + 1 - len(pos[::BLOCK_SYMBOLS][:nblocks])))
    is_m = sym >= 256
    lc = np.where(is_m, sym - 256, 0)
    lcode = LENGTH_CODE[lc]
    lsym = np.where(is_m, 257 + lcode, sym)
    xlen = np.where(is_m, np.array(EXTRA_LBITS, np.int64)[lcode], 0)
    xval = np.where(xlen > 0, lc - BASE_LENGTH[lcode], 0)        # code 285 (length 258) sends no extra bits
    pieces = []                                       # finished whole bytes
    carry_v, carry_n = 0, 0                           # < 8 pending bits
    for b in range(nblocks):
        a, e = b * BLOCK_SYMBOLS, min((b + 1) * BLOCK_SYMBOLS, T)
        last = int(b == nblocks - 1)
        freq = np.bincount(lsym[a:e], minlength=L_CODES)
        freq[END_BLOCK] += 1
        nm = int(is_m[a:e].sum())
        stored_len = int(bstart[b + 1] - bstart[b])
        kind, llen, lcd, dlen, dcd, header = block_plan(freq.tolist(), nm, stored_len)
        if kind == 0:
            v = carry_v | (last << carry_n)           # STORED_BLOCK << 1 | last, then bi_windup
            n = carry_n + 3
            pieces.append(np.frombuffer(int(v).to_bytes((n + 7) >> 3, "little"), np.uint8))
            pieces.append(np.frombuffer(struct.pack("<HH", stored_len, stored_len ^ 0xFFFF), np.uint8))
            pieces.append(f[bstart[b]:bstart[b + 1]])
            carry_v, carry_n = 0, 0
            continue
        vl, ll = [carry_v, (kind << 1) | last], [carry_n, 3]
        if header:
            vl += [h[0] for h in header]
            ll += [h[1] for h in header]
        llen, lcd = np.array(llen, np.int64), np.array(lcd, np.int64)
        s = lsym[a:e]
        cv = lcd[s]
        cl = llen[s]
        # code, then extra bits, then the distance code (0 extra bits) for matches: one (value, length) per symbol
        dv, dl = int(dcd[0]), int(dlen[0])
        mm = is_m[a:e]
        v = cv | (xval[a:e] << cl) | np.where(mm, dv << (cl + xlen[a:e]), 0)
        ln = cl + xlen[a:e] + np.where(mm, dl, 0)
        vl = np.concatenate([np.array(vl, np.int64), v, [lcd[END_BLOCK]]])
        ll = np.concatenate([np.array(ll, np.int64), ln, [llen[END_BLOCK]]])
        data, endbit = _pack(vl, ll, 0)
        full = endbit >> 3
        pieces.append(data[:full])
        carry_n = endbit & 7
        carry_v = int(data[full]) if carry_n else 0
    if carry_n:
        pieces.append(np.array([carry_v], np.uint8))   # bi_windup after the last block
    return np.concatenate(pieces).tobytes()


def adler32(f: np.ndarray) -> int:
    n = f.size
    x = f.astype(np.int64)
    a = (1 + int(x.sum())) % 65521
    b = (n + int(((n - np.arange(n, dtype=np.int64)) * x).sum() % 65521)) % 65521
    return (b << 16) | a


def zlib_header(data_size: int) -> bytes:
    """zlib's 78 01 (window 32K, FLEVEL 0), then libpng's optimize_cmf for data_size <= 16384."""
    cmf, flg = 0x78, 0x01
    if data_size <= 16384:
        cinfo = cmf >> 4
        half = 1 << (cinfo + 7)
        if data_size <= half:
            while True:
                half >>= 1
                cinfo -= 1
                if not (cinfo > 0 and data_size <= half):
                    break
            cmf = (cmf & 0x0F) | (cinfo << 4)
            tmp = flg & 0xE0
            tmp += 0x1F - ((cmf << 8) + tmp) % 0x1F
            flg = tmp
    return bytes([cmf, flg])


def _chunk(kind: bytes, payload: bytes) -> bytes:
    return struct.pack(">I", len(payload)) + kind + payload + struct.pack(">I", _zlib_crc.crc32(kind + payload))


def header(H: int, W: int) -> bytes:
    """Signature, IHDR, and the zlib CMF / FLG that open the first IDAT payload."""
    ihdr = struct.pack(">IIBBBBB", W, H, 8, 2, 0, 0, 0)
    return SIGNATURE + _chunk(b"IHDR", ihdr) + zlib_header(H * (3 * W + 1))


def idat_chunks(z: bytes) -> bytes:
    return b"".join(_chunk(b"IDAT", z[i:i + IDAT_PAYLOAD]) for i in range(0, len(z), IDAT_PAYLOAD))


def imencode(bgr: np.ndarray) -> bytes:
    """What cv2.imencode(".png", bgr) returns, as bytes."""
    assert bgr.ndim == 3 and bgr.shape[2] == 3 and bgr.dtype == np.uint8
    H, W, _ = bgr.shape
    f = filtered(bgr)
    hdr = header(H, W)
    z = hdr[-2:] + deflate(f) + struct.pack(">I", adler32(f))
    return hdr[:-2] + idat_chunks(z) + _chunk(b"IEND", b"")
