// K10 -- batched PNG encoder, byte-identical to cv2.imencode(".png") with OpenCV's defaults (libpng 1.6 + zlib:
// filter Sub, deflate level 1 with strategy Z_RLE, memLevel 8, IDAT payloads of 8192 bytes).  oracle/png.py is the
// NumPy statement of the same stages; DESIGN.md "K10" carries the format facts and the parse argument.
//   png_filter       one CTA per 4096 filtered bytes: BGR -> RGB, Sub filter, filter-type bytes; writes the filtered
//                    stream, the first / last run boundary of the tile and the tile's Adler-32 partial sums
//   png_run_carry    one CTA per frame: start of the run open at each tile's start, end of the run open at its end
//   png_symbols      (twice) per tile: deflate_rle's symbol starts in closed form from the run containing each byte;
//                    the first pass counts symbols per tile, the second writes them at their stream index and records
//                    where every 16383-symbol block starts
//   png_sym_scan     one CTA per frame: exclusive scan of tile symbol counts, symbol and block totals
//   png_block_plan   one CTA per deflate block: histogram, then one thread restates trees.c (build_tree, gen_bitlen,
//                    gen_codes, scan_tree / send_tree) and _tr_flush_block's stored / static / dynamic choice
//   png_block_scan   one CTA per frame: bit offset of every block (stored blocks align to a byte), stream length
//   png_zero         clears exactly the words the frame's deflate bits occupy
//   png_emit         one CTA per block: tree description by one thread, symbols by all (atomicOr on shared words),
//                    stored blocks copied byte-aligned
//   png_frame        one CTA per IDAT chunk: signature + IHDR, zlib header, data, Adler-32, chunk framing with CRC-32
//                    (per-thread CRCs joined with crc32_combine), IEND
#include <string.h>

#include "avb_common.cuh"

namespace {

constexpr int THREADS = 256;
constexpr int PER_THREAD = 16;
constexpr int TILE = THREADS * PER_THREAD;       // filtered bytes per tile
constexpr int BLOCK_SYMBOLS = 16383;             // zlib lit_bufsize - 1 (memLevel 8)
constexpr int MAX_MATCH = 258;
constexpr int IDAT = 8192;                       // libpng zbuffer size
constexpr int L_CODES = 286, D_CODES = 30, BL_CODES = 19, END_BLOCK = 256;
constexpr int HEAP_SIZE = 2 * L_CODES + 1;
// A tree description is 5 + 5 + 4 + 19 * 3 bits, then at most 286 + 30 code-length symbols of <= 7 + 7 bits.
constexpr int HDR_WORDS = (14 + 57 + (L_CODES + D_CODES) * 14 + 31) / 32;
constexpr int64_t ADLER_MOD = 65521;
constexpr int SIG_IHDR = 33;                     // signature (8) + IHDR chunk (25)

__constant__ uint8_t c_extra_lbits[29] = {0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0};
__constant__ uint8_t c_no_dextra[30] = {0};     // only distance 1 (code 0) occurs
__constant__ uint8_t c_extra_blbits[19] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 2, 3, 7};
__constant__ uint8_t c_bl_order[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};

struct LenTabs {
    uint8_t code[256];      // trees.c _length_code[len - 3]
    uint8_t base[29];       // base_length[code]
};
constexpr LenTabs make_len_tabs() {
    LenTabs t{};
    constexpr uint8_t ex[29] = {0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0};
    int length = 0;
    for (int code = 0; code < 28; ++code) {
        t.base[code] = (uint8_t)length;
        for (int i = 0; i < (1 << ex[code]); ++i) t.code[length++] = (uint8_t)code;
    }
    t.code[length - 1] = 28;
    return t;
}
__constant__ LenTabs c_len = make_len_tabs();

struct CrcTabs {
    uint32_t t[256];
    uint32_t x2n[32];       // x^(2^k) mod p, zlib crc32.c x2n_table
};
constexpr uint32_t multmodp_c(uint32_t a, uint32_t b) {
    uint32_t m = 1u << 31, p = 0;
    for (;;) {
        if (a & m) {
            p ^= b;
            if ((a & (m - 1)) == 0) break;
        }
        m >>= 1;
        b = b & 1 ? (b >> 1) ^ 0xEDB88320u : b >> 1;
    }
    return p;
}
constexpr CrcTabs make_crc() {
    CrcTabs c{};
    for (uint32_t n = 0; n < 256; ++n) {
        uint32_t v = n;
        for (int k = 0; k < 8; ++k) v = v & 1 ? (v >> 1) ^ 0xEDB88320u : v >> 1;
        c.t[n] = v;
    }
    uint32_t p = 1u << 30;  // x^1
    c.x2n[0] = p;
    for (int k = 1; k < 32; ++k) c.x2n[k] = p = multmodp_c(p, p);
    return c;
}
__constant__ CrcTabs c_crc = make_crc();

__device__ __forceinline__ uint32_t multmodp(uint32_t a, uint32_t b) {
    uint32_t m = 1u << 31, p = 0;
    for (;;) {
        if (a & m) {
            p ^= b;
            if ((a & (m - 1)) == 0) break;
        }
        m >>= 1;
        b = b & 1 ? (b >> 1) ^ 0xEDB88320u : b >> 1;
    }
    return p;
}
// crc32_combine: the CRC of A || B from crc(A), crc(B) and len(B)
__device__ uint32_t crc_combine(uint32_t c1, uint32_t c2, uint32_t len2) {
    uint32_t p = 1u << 31;
    for (int k = 3; len2; len2 >>= 1, ++k)
        if (len2 & 1) p = multmodp(c_crc.x2n[k & 31], p);
    return multmodp(p, c1) ^ c2;
}

struct Geo {
    int H, W;
    int64_t S;              // filtered bytes per frame: H * (3W + 1)
    int64_t Sp;             // S rounded up to 16
    int64_t ntiles;
    int64_t maxb;           // blocks per frame at most: S / 16383 + 1, plus the sentinel start
    int64_t wwords;         // deflate staging words per frame
    int64_t maxchunks;      // IDAT chunks per frame at most
};

// per-frame totals
struct Frame {
    unsigned long long s1, s2;   // Adler-32 sums (each tile adds its partials reduced mod 65521)
    int64_t T;                   // symbols
    int64_t nblocks;
    int64_t bits;                // deflate bits
    int64_t zlen;                // zlib stream bytes
    int64_t nchunks;
    int64_t pad;
};

struct Plan {
    uint32_t code[L_CODES];  // (len << 16) | bit-reversed code
    uint32_t dist;           // distance code 0
    uint32_t kind;           // 0 stored, 1 static, 2 dynamic
    uint32_t hdr_bits;       // tree description bits (dynamic)
    uint32_t pad;
    uint64_t body_bits;      // 3 + tree description + data + end of block (Huffman); stored: the payload bytes
    uint32_t hdr[HDR_WORDS];
};

struct Work {
    uint8_t *F;              // [n][Sp] filtered bytes
    int64_t *tfirst, *tlast; // [n][ntiles] first / last run boundary in the tile (S / -1 when none)
    int64_t *tcnt;           // [n][ntiles] symbols, then their exclusive offsets
    uint16_t *syms;          // [n][S] <256 literal, 256 + len - 3 match
    int64_t *bstart;         // [n][maxb] first filtered byte of each block, sentinel S
    uint64_t *boff;          // [n][maxb] bit offset of each block
    Plan *plan;              // [n][maxb]
    Frame *fr;               // [n]
    uint32_t *words;         // [n][wwords]
};

int64_t align16(int64_t x) { return (x + 15) & ~(int64_t)15; }

Geo geometry(int H, int W) {
    Geo g;
    g.H = H;
    g.W = W;
    g.S = (int64_t)H * (3LL * W + 1);
    g.Sp = align16(g.S);
    g.ntiles = (g.S + TILE - 1) / TILE;
    g.maxb = g.S / BLOCK_SYMBOLS + 2;
    // Every block costs at most its static form (<= 9 bits per byte + 10 bits) or its stored form; see DESIGN.md K10.
    const int64_t dbits = 9 * g.S + 48 * g.maxb + 8;
    g.wwords = (dbits + 31) / 32 + 2;
    const int64_t zmax = (dbits + 7) / 8 + 6;
    g.maxchunks = zmax / IDAT + 1;
    return g;
}

int64_t carve(const Geo &g, int n, uint8_t *base, Work *w) {
    int64_t off = 0;
    auto take = [&](int64_t bytes) {
        uint8_t *p = base ? base + off : nullptr;
        off += align16(bytes);
        return p;
    };
    uint8_t *F = take(n * g.Sp);
    uint8_t *tf = take(n * g.ntiles * 8), *tl = take(n * g.ntiles * 8), *tc = take(n * g.ntiles * 8);
    uint8_t *sy = take(n * g.S * 2);
    uint8_t *bs = take(n * g.maxb * 8), *bo = take(n * g.maxb * 8);
    uint8_t *pl = take(n * g.maxb * (int64_t)sizeof(Plan));
    uint8_t *fr = take(n * (int64_t)sizeof(Frame));
    uint8_t *wd = take(n * g.wwords * 4);
    if (w) {
        w->F = F;
        w->tfirst = (int64_t *)tf;
        w->tlast = (int64_t *)tl;
        w->tcnt = (int64_t *)tc;
        w->syms = (uint16_t *)sy;
        w->bstart = (int64_t *)bs;
        w->boff = (uint64_t *)bo;
        w->plan = (Plan *)pl;
        w->fr = (Frame *)fr;
        w->words = (uint32_t *)wd;
    }
    return off;
}

// ------------------------------------------------------------------------------------------------ block scans
// Inclusive scan over the CTA of one value per thread with an associative op; returns the inclusive value and sets
// *total to the reduction of all threads.
template <class T, class Op>
__device__ T cta_scan(T x, T ident, Op op, T *total) {
    __shared__ T wsum[THREADS / 32];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const T y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o) x = op(y, x);
    }
    if (lane == 31) wsum[wid] = x;
    __syncthreads();
    if (wid == 0) {
        T t = lane < THREADS / 32 ? wsum[lane] : ident;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const T y = __shfl_up_sync(0xffffffffu, t, o);
            if (lane >= o) t = op(y, t);
        }
        if (lane < THREADS / 32) wsum[lane] = t;
    }
    __syncthreads();
    if (wid) x = op(wsum[wid - 1], x);
    *total = wsum[THREADS / 32 - 1];
    __syncthreads();
    return x;
}

struct OpMax {
    __device__ int64_t operator()(int64_t a, int64_t b) const { return a > b ? a : b; }
};
struct OpMin {
    __device__ int64_t operator()(int64_t a, int64_t b) const { return a < b ? a : b; }
};
struct OpAdd {
    __device__ int64_t operator()(int64_t a, int64_t b) const { return a + b; }
};

// ------------------------------------------------------------------------------------------------ png_filter
__global__ void __launch_bounds__(THREADS) png_filter_kernel(const uint8_t *in, int64_t fs, int64_t rs, Geo g, Work w) {
    const int f = blockIdx.y;
    const int64_t t = blockIdx.x, p0 = t * TILE + (int64_t)threadIdx.x * PER_THREAD;
    const uint8_t *fin = in + (int64_t)f * fs;
    const int64_t rowb = 3LL * g.W + 1;
    const uint8_t ftype = g.W > 1 ? 1 : 0;
    auto fbyte = [&](int64_t y, int64_t c) -> uint8_t {
        if (c == 0) return ftype;
        const int64_t i = c - 1, px = i / 3;
        const int ch = 2 - (int)(i - px * 3);
        const uint8_t *row = fin + y * rs;
        const uint8_t x = row[px * 3 + ch];
        return px ? (uint8_t)(x - row[(px - 1) * 3 + ch]) : x;
    };
    uint8_t v[PER_THREAD];
    int64_t first = g.S, last = -1;
    uint64_t s1 = 0, s2 = 0;
    if (p0 < g.S) {
        int64_t y = p0 / rowb, c = p0 - y * rowb;
        uint8_t prev = 0;
        if (p0 > 0) prev = c ? fbyte(y, c - 1) : fbyte(y - 1, rowb - 1);
        for (int k = 0; k < PER_THREAD; ++k) {
            const int64_t p = p0 + k;
            if (p >= g.S) {
                v[k] = 0;
                continue;
            }
            const uint8_t b = fbyte(y, c);
            v[k] = b;
            if (p == 0 || b != prev) {
                if (first == g.S) first = p;
                last = p;
            }
            prev = b;
            s1 += b;
            s2 += (uint64_t)(g.S - p) % ADLER_MOD * b;
            if (++c == rowb) c = 0, ++y;
        }
        uint4 q;
        memcpy(&q, v, 16);
        *reinterpret_cast<uint4 *>(w.F + (int64_t)f * g.Sp + p0) = q;
    }
    int64_t tot;
    cta_scan<int64_t>(first, g.S, OpMin(), &tot);
    if (threadIdx.x == 0) w.tfirst[(int64_t)f * g.ntiles + t] = tot;
    cta_scan<int64_t>(last, -1, OpMax(), &tot);
    if (threadIdx.x == 0) w.tlast[(int64_t)f * g.ntiles + t] = tot;
    cta_scan<int64_t>((int64_t)(s1 % ADLER_MOD), 0, OpAdd(), &tot);
    int64_t tot2;
    cta_scan<int64_t>((int64_t)(s2 % ADLER_MOD), 0, OpAdd(), &tot2);
    if (threadIdx.x == 0) {
        atomicAdd(&w.fr[f].s1, (unsigned long long)(tot % ADLER_MOD));
        atomicAdd(&w.fr[f].s2, (unsigned long long)(tot2 % ADLER_MOD));
    }
}

// ------------------------------------------------------------------------------------------------ png_run_carry
// tlast[t] becomes the start of the run open at tile t's first byte (the last boundary before the tile), tfirst[t]
// the end of the run open at its last byte (the first boundary after the tile, or S).
__global__ void __launch_bounds__(THREADS) png_run_carry_kernel(Geo g, Work w) {
    const int f = blockIdx.x;
    int64_t *tl = w.tlast + (int64_t)f * g.ntiles, *tf = w.tfirst + (int64_t)f * g.ntiles;
    __shared__ int64_t inc[THREADS];
    int64_t carry = -1, tot;
    for (int64_t base = 0; base < g.ntiles; base += THREADS) {
        const int64_t i = base + threadIdx.x;
        inc[threadIdx.x] = cta_scan<int64_t>(i < g.ntiles ? tl[i] : -1, -1, OpMax(), &tot);
        __syncthreads();
        if (i < g.ntiles) tl[i] = threadIdx.x ? max(carry, inc[threadIdx.x - 1]) : carry;
        carry = max(carry, tot);
        __syncthreads();
    }
    carry = g.S;                                   // reversed: thread k of a chunk takes tile base + THREADS-1-k
    for (int64_t base = (g.ntiles - 1) / THREADS * THREADS; base >= 0; base -= THREADS) {
        const int64_t i = base + THREADS - 1 - threadIdx.x;
        inc[threadIdx.x] = cta_scan<int64_t>(i < g.ntiles ? tf[i] : g.S, g.S, OpMin(), &tot);
        __syncthreads();
        if (i < g.ntiles) tf[i] = threadIdx.x ? min(carry, inc[threadIdx.x - 1]) : carry;
        carry = min(carry, tot);
        __syncthreads();
    }
}

// ------------------------------------------------------------------------------------------------ png_symbols
// Symbol at byte p of a run [rs, re): the closed form of deflate_rle (oracle/png.py parse).  Returns -1 when p only
// continues a match, else the symbol code (<256 literal, 256 + len - 3 match).
__device__ __forceinline__ int symbol_at(int64_t p, int64_t rs, int64_t re, uint8_t b) {
    const int64_t o = p - rs;
    if (o == 0) return b;
    const int64_t q = o - 1, R1 = re - rs - 1;
    const int64_t m = R1 / MAX_MATCH, r = R1 - m * MAX_MATCH;
    if (q < m * MAX_MATCH) return (q % MAX_MATCH) == 0 ? 256 + MAX_MATCH - 3 : -1;
    if (r >= 3) return q == m * MAX_MATCH ? 256 + (int)r - 3 : -1;
    return b;
}

template <bool WRITE>
__global__ void __launch_bounds__(THREADS) png_symbols_kernel(Geo g, Work w) {
    const int f = blockIdx.y;
    const int64_t t = blockIdx.x, p0 = t * TILE + (int64_t)threadIdx.x * PER_THREAD;
    const uint8_t *F = w.F + (int64_t)f * g.Sp;
    const int64_t ft = (int64_t)f * g.ntiles + t;
    uint8_t v[PER_THREAD];
    {
        const uint4 q = *reinterpret_cast<const uint4 *>(F + min(p0, g.Sp - 16));
        memcpy(v, &q, 16);
    }
    const int nk = (int)max((int64_t)0, min((int64_t)PER_THREAD, g.S - p0));
    const uint8_t prev = p0 > 0 && p0 < g.S ? F[p0 - 1] : 0;
    int64_t first = g.S, last = -1;
    for (int k = 0; k < nk; ++k) {
        const int64_t p = p0 + k;
        if (p == 0 || v[k] != (k ? v[k - 1] : prev)) {
            if (first == g.S) first = p;
            last = p;
        }
    }
    int64_t tot;
    // run start at this thread's first byte: max boundary before it
    const int64_t incl = cta_scan<int64_t>(last, -1, OpMax(), &tot);
    int64_t rs = __shfl_up_sync(0xffffffffu, incl, 1);
    {
        __shared__ int64_t wl[THREADS / 32];
        if ((threadIdx.x & 31) == 31) wl[threadIdx.x >> 5] = incl;
        __syncthreads();
        if ((threadIdx.x & 31) == 0) rs = threadIdx.x ? wl[(threadIdx.x >> 5) - 1] : -1;
        __syncthreads();
    }
    rs = max(rs, w.tlast[ft]);
    // run end after this thread's last byte: min boundary after it (reverse scan through thread order)
    const int64_t ridx = THREADS - 1 - threadIdx.x;
    int64_t re;
    {
        __shared__ int64_t firsts[THREADS];
        firsts[threadIdx.x] = first;
        __syncthreads();
        const int64_t mine = firsts[ridx];
        __syncthreads();
        const int64_t inc = cta_scan<int64_t>(mine, g.S, OpMin(), &tot);   // over reversed order
        firsts[ridx] = inc;                                                  // min of firsts[ridx..]
        __syncthreads();
        re = threadIdx.x + 1 < THREADS ? firsts[threadIdx.x + 1] : g.S;
        __syncthreads();
    }
    re = min(re, w.tfirst[ft]);
    // per byte: run start forward, run end backward
    int64_t rend[PER_THREAD];
    {
        int64_t e = re;
        for (int k = PER_THREAD - 1; k >= 0; --k) {
            rend[k] = e;
            if (k < nk && (p0 + k == 0 || v[k] != (k ? v[k - 1] : prev))) e = p0 + k;
        }
    }
    int sym[PER_THREAD];
    int cnt = 0;
    for (int k = 0; k < PER_THREAD; ++k) {
        sym[k] = -1;
        if (k >= nk) continue;
        const int64_t p = p0 + k;
        if (p == 0 || v[k] != (k ? v[k - 1] : prev)) rs = p;
        sym[k] = symbol_at(p, rs, rend[k], v[k]);
        cnt += sym[k] >= 0;
    }
    const int64_t cincl = cta_scan<int64_t>(cnt, 0, OpAdd(), &tot);
    if (!WRITE) {
        if (threadIdx.x == 0) w.tcnt[ft] = tot;
        return;
    }
    int64_t gi = w.tcnt[ft] + cincl - cnt;
    uint16_t *syms = w.syms + (int64_t)f * g.S;
    int64_t *bstart = w.bstart + (int64_t)f * g.maxb;
    for (int k = 0; k < nk; ++k) {
        if (sym[k] < 0) continue;
        syms[gi] = (uint16_t)sym[k];
        if (gi % BLOCK_SYMBOLS == 0) bstart[gi / BLOCK_SYMBOLS] = p0 + k;
        ++gi;
    }
}

__global__ void __launch_bounds__(THREADS) png_sym_scan_kernel(Geo g, Work w) {
    const int f = blockIdx.x;
    int64_t *c = w.tcnt + (int64_t)f * g.ntiles;
    int64_t carry = 0;
    for (int64_t base = 0; base < g.ntiles; base += THREADS) {
        const int64_t i = base + threadIdx.x;
        const int64_t x = i < g.ntiles ? c[i] : 0;
        int64_t tot;
        const int64_t inc = cta_scan<int64_t>(x, 0, OpAdd(), &tot);
        if (i < g.ntiles) c[i] = carry + inc - x;
        carry += tot;
    }
    if (threadIdx.x == 0) {
        const int64_t T = carry, nb = T / BLOCK_SYMBOLS + 1;
        w.fr[f].T = T;
        w.fr[f].nblocks = nb;
        int64_t *bstart = w.bstart + (int64_t)f * g.maxb;
        if (T % BLOCK_SYMBOLS == 0) bstart[nb - 1] = g.S;   // Z_FINISH's empty final block
        bstart[nb] = g.S;
    }
}

// ------------------------------------------------------------------------------------------------ trees.c
struct TreeSmem {
    int freq[HEAP_SIZE];
    int len[HEAP_SIZE];     // Len of leaves and, while building, of internal nodes
    int dad[HEAP_SIZE];
    int heap[HEAP_SIZE];
    uint8_t depth[HEAP_SIZE];
    int bl_count[16];
    int next_code[16];
};

struct Acc {
    int64_t opt_len, static_len;
};

__device__ __forceinline__ bool smaller(const TreeSmem &s, int n, int m) {
    return s.freq[n] < s.freq[m] || (s.freq[n] == s.freq[m] && s.depth[n] <= s.depth[m]);
}

__device__ void downheap(TreeSmem &s, int heap_len, int k) {
    const int v = s.heap[k];
    int j = k << 1;
    while (j <= heap_len) {
        if (j < heap_len && smaller(s, s.heap[j + 1], s.heap[j])) ++j;
        if (smaller(s, v, s.heap[j])) break;
        s.heap[k] = s.heap[j];
        k = j;
        j <<= 1;
    }
    s.heap[k] = v;
}

__device__ __forceinline__ uint32_t bi_reverse(uint32_t code, int len) { return __brev(code) >> (32 - len); }

// build_tree + gen_bitlen + gen_codes over s.freq[0..elems); static lengths slen (null for the bit-length tree).
// Leaves' (len << 16) | code go to out[0..elems).  Returns max_code.
__device__ int build_tree(TreeSmem &s, int elems, int max_length, int extra_base, const uint8_t *extra,
                          int (*slen)(int), Acc &acc, uint32_t *out) {
    int heap_len = 0, heap_max = HEAP_SIZE, max_code = -1;
    for (int n = 0; n < elems; ++n) {
        if (s.freq[n]) {
            s.heap[++heap_len] = max_code = n;
            s.depth[n] = 0;
        } else {
            s.len[n] = 0;
        }
    }
    while (heap_len < 2) {
        const int node = s.heap[++heap_len] = (max_code < 2 ? ++max_code : 0);
        s.freq[node] = 1;
        s.depth[node] = 0;
        acc.opt_len--;
        if (slen) acc.static_len -= slen(node);
    }
    for (int n = heap_len / 2; n >= 1; --n) downheap(s, heap_len, n);
    int node = elems;
    do {
        const int n = s.heap[1];
        s.heap[1] = s.heap[heap_len--];
        downheap(s, heap_len, 1);
        const int m = s.heap[1];
        s.heap[--heap_max] = n;
        s.heap[--heap_max] = m;
        s.freq[node] = s.freq[n] + s.freq[m];
        s.depth[node] = (uint8_t)((s.depth[n] >= s.depth[m] ? s.depth[n] : s.depth[m]) + 1);
        s.dad[n] = s.dad[m] = node;
        s.heap[1] = node++;
        downheap(s, heap_len, 1);
    } while (heap_len >= 2);
    s.heap[--heap_max] = s.heap[1];
    // gen_bitlen
    for (int b = 0; b < 16; ++b) s.bl_count[b] = 0;
    s.len[s.heap[heap_max]] = 0;
    int overflow = 0, h;
    for (h = heap_max + 1; h < HEAP_SIZE; ++h) {
        const int n = s.heap[h];
        int bits = s.len[s.dad[n]] + 1;
        if (bits > max_length) bits = max_length, ++overflow;
        s.len[n] = bits;
        if (n > max_code) continue;
        s.bl_count[bits]++;
        const int xbits = n >= extra_base ? extra[n - extra_base] : 0;
        const int64_t fq = s.freq[n];
        acc.opt_len += fq * (bits + xbits);
        if (slen) acc.static_len += fq * (slen(n) + xbits);
    }
    if (overflow) {
        do {
            int bits = max_length - 1;
            while (s.bl_count[bits] == 0) bits--;
            s.bl_count[bits]--;
            s.bl_count[bits + 1] += 2;
            s.bl_count[max_length]--;
            overflow -= 2;
        } while (overflow > 0);
        for (int bits = max_length; bits != 0; bits--) {
            int n = s.bl_count[bits];
            while (n != 0) {
                const int m = s.heap[--h];
                if (m > max_code) continue;
                if (s.len[m] != bits) {
                    acc.opt_len += ((int64_t)bits - s.len[m]) * s.freq[m];
                    s.len[m] = bits;
                }
                n--;
            }
        }
    }
    // gen_codes
    int code = 0;
    for (int bits = 1; bits <= 15; ++bits) s.next_code[bits] = code = (code + s.bl_count[bits - 1]) << 1;
    for (int n = 0; n < elems; ++n) {
        const int ln = n <= max_code ? s.len[n] : 0;
        out[n] = ln ? ((uint32_t)ln << 16) | bi_reverse((uint32_t)s.next_code[ln]++, ln) : 0u;
    }
    return max_code;
}

__device__ int static_llen(int n) { return n < 144 ? 8 : n < 256 ? 9 : n < 280 ? 7 : 8; }
__device__ int static_dlen(int) { return 5; }
__device__ uint32_t static_lcode(int n) {
    // gen_codes over the fixed lengths: 7-bit codes 0..23 for 256..279, 8-bit 48.. for 0..143, 192.. for 280..287,
    // 9-bit 400.. for 144..255
    if (n < 144) return (8u << 16) | bi_reverse(48 + n, 8);
    if (n < 256) return (9u << 16) | bi_reverse(400 + n - 144, 9);
    if (n < 280) return (7u << 16) | bi_reverse(n - 256, 7);
    return (8u << 16) | bi_reverse(192 + n - 280, 8);
}

// scan_tree (count) / send_tree (emit) over lens of codes[0..max_code]
template <class Sink>
__device__ void tree_runs(const uint32_t *codes, int max_code, Sink sink) {
    int prevlen = -1, nextlen = (int)(codes[0] >> 16), count = 0;
    int max_count = 7, min_count = 4;
    if (nextlen == 0) max_count = 138, min_count = 3;
    for (int n = 0; n <= max_code; ++n) {
        const int curlen = nextlen;
        nextlen = n + 1 <= max_code ? (int)(codes[n + 1] >> 16) : 0xffff;
        if (++count < max_count && curlen == nextlen) continue;
        if (count < min_count) {
            do sink(curlen, 0, 0);
            while (--count != 0);
        } else if (curlen != 0) {
            if (curlen != prevlen) {
                sink(curlen, 0, 0);
                count--;
            }
            sink(16, count - 3, 2);
        } else if (count <= 10) {
            sink(17, count - 3, 3);
        } else {
            sink(18, count - 11, 7);
        }
        count = 0;
        prevlen = curlen;
        if (nextlen == 0) max_count = 138, min_count = 3;
        else if (curlen == nextlen) max_count = 6, min_count = 3;
        else max_count = 7, min_count = 4;
    }
}

struct HdrWriter {
    uint32_t *hdr;
    uint32_t n = 0;
    __device__ void put(uint32_t v, int len) {
        for (int i = 0; i < len; ++i, ++n)
            if ((v >> i) & 1) hdr[n >> 5] |= 1u << (n & 31);
    }
};

__global__ void __launch_bounds__(THREADS) png_block_plan_kernel(Geo g, Work w) {
    const int f = blockIdx.y;
    const int64_t b = blockIdx.x;
    const Frame &fr = w.fr[f];
    if (b >= fr.nblocks) return;
    __shared__ TreeSmem s;
    __shared__ int hist[L_CODES];
    __shared__ int nmatch;
    __shared__ uint32_t lt[L_CODES], dt[D_CODES], bt[BL_CODES], hsh[HDR_WORDS];
    for (int i = threadIdx.x; i < L_CODES; i += THREADS) hist[i] = 0;
    if (threadIdx.x == 0) nmatch = 0;
    __syncthreads();
    const int64_t a = b * BLOCK_SYMBOLS, e = min(a + BLOCK_SYMBOLS, fr.T);
    const uint16_t *syms = w.syms + (int64_t)f * g.S;
    int nm = 0;
    for (int64_t i = a + threadIdx.x; i < e; i += THREADS) {
        const int sy = syms[i];
        if (sy < 256) {
            atomicAdd(&hist[sy], 1);
        } else {
            atomicAdd(&hist[257 + c_len.code[sy - 256]], 1);
            ++nm;
        }
    }
    atomicAdd(&nmatch, nm);
    __syncthreads();
    if (threadIdx.x != 0) return;
    Plan &P = w.plan[(int64_t)f * g.maxb + b];
    const int64_t *bstart = w.bstart + (int64_t)f * g.maxb;
    const int64_t stored_len = bstart[b + 1] - bstart[b];
    Acc acc{0, 0};
    hist[END_BLOCK] += 1;
    for (int i = 0; i < L_CODES; ++i) s.freq[i] = hist[i];
    const int lmax = build_tree(s, L_CODES, 15, 257, c_extra_lbits, static_llen, acc, lt);
    s.freq[0] = nmatch;
    for (int i = 1; i < D_CODES; ++i) s.freq[i] = 0;
    const int dmax = build_tree(s, D_CODES, 15, 0, c_no_dextra, static_dlen, acc, dt);
    for (int i = 0; i < BL_CODES; ++i) s.freq[i] = 0;
    auto count = [&](int sym, int, int) { s.freq[sym]++; };
    tree_runs(lt, lmax, count);
    tree_runs(dt, dmax, count);
    build_tree(s, BL_CODES, 7, 0, c_extra_blbits, nullptr, acc, bt);
    int max_blindex;
    for (max_blindex = BL_CODES - 1; max_blindex >= 3; max_blindex--)
        if (bt[c_bl_order[max_blindex]] >> 16) break;
    acc.opt_len += 3 * ((int64_t)max_blindex + 1) + 5 + 5 + 4;
    int64_t opt_lenb = (acc.opt_len + 3 + 7) >> 3;
    const int64_t static_lenb = (acc.static_len + 3 + 7) >> 3;
    if (static_lenb <= opt_lenb) opt_lenb = static_lenb;
    if (stored_len + 4 <= opt_lenb) {
        P.kind = 0;
        P.body_bits = (uint64_t)stored_len;
        return;
    }
    const bool stat = static_lenb == opt_lenb;
    P.kind = stat ? 1 : 2;
    for (int i = 0; i < L_CODES; ++i) P.code[i] = stat ? static_lcode(i) : lt[i];
    P.dist = stat ? ((5u << 16) | 0u) : dt[0];
    uint64_t bits = 3;
    if (!stat) {
        for (int i = 0; i < HDR_WORDS; ++i) hsh[i] = 0;
        HdrWriter hw{hsh};
        hw.put((uint32_t)(lmax + 1 - 257), 5);
        hw.put((uint32_t)(dmax + 1 - 1), 5);
        hw.put((uint32_t)(max_blindex + 1 - 4), 4);
        for (int r = 0; r <= max_blindex; ++r) hw.put(bt[c_bl_order[r]] >> 16, 3);
        auto send = [&](int sym, int v, int nb) {
            hw.put(bt[sym] & 0xffffu, (int)(bt[sym] >> 16));
            if (nb) hw.put((uint32_t)v, nb);
        };
        tree_runs(lt, lmax, send);
        tree_runs(dt, dmax, send);
        P.hdr_bits = hw.n;
        for (uint32_t i = 0; i < (hw.n + 31) / 32; ++i) P.hdr[i] = hsh[i];
        bits += hw.n;
    } else {
        P.hdr_bits = 0;
    }
    for (int i = 0; i < L_CODES; ++i) {
        const int fq = hist[i];
        if (!fq) continue;
        const int xb = i >= 257 ? c_extra_lbits[i - 257] : 0;
        bits += (uint64_t)fq * ((P.code[i] >> 16) + xb);
    }
    bits += (uint64_t)nmatch * (P.dist >> 16);
    P.body_bits = bits;
}

__global__ void __launch_bounds__(THREADS) png_block_scan_kernel(Geo g, Work w) {
    const int f = blockIdx.x;
    Frame &fr = w.fr[f];
    const int64_t nb = fr.nblocks;
    const Plan *P = w.plan + (int64_t)f * g.maxb;
    const int64_t *bstart = w.bstart + (int64_t)f * g.maxb;
    uint64_t *boff = w.boff + (int64_t)f * g.maxb;
    // Block b maps bit offset x to x + a (Huffman) or align8(x + 3) + d (stored, d a multiple of 8).  Both forms
    // compose into one of the two, because align8(align8(y) + e) = align8(y) + align8(e): scan those maps.
    struct M {
        int64_t c, d;       // align8(x + c) + d when c >= 0, else x + d
    };
    auto compose = [](M p, M q) -> M {     // q after p
        if (q.c < 0) return M{p.c, p.d + q.d};
        if (p.c < 0) return M{p.d + q.c, q.d};
        return M{p.c, ((p.d + q.c + 7) & ~7LL) + q.d};
    };
    uint64_t carry = 0;
    for (int64_t base = 0; base < nb; base += THREADS) {
        const int64_t i = base + threadIdx.x;
        M m{-1, 0};
        if (i < nb) {
            if (P[i].kind == 0) m = M{3, 32 + 8 * (bstart[i + 1] - bstart[i])};
            else m = M{-1, (int64_t)P[i].body_bits};
        }
        // inclusive scan with the composition (lanes, then warps)
        __shared__ int64_t wc[THREADS / 32], wd[THREADS / 32];
        const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
        M x = m;
        for (int o = 1; o < 32; o <<= 1) {
            M y{__shfl_up_sync(0xffffffffu, x.c, o), __shfl_up_sync(0xffffffffu, x.d, o)};
            if (lane >= o) x = compose(y, x);
        }
        if (lane == 31) wc[wid] = x.c, wd[wid] = x.d;
        __syncthreads();
        if (threadIdx.x == 0)
            for (int k = 1; k < THREADS / 32; ++k) {
                const M r = compose(M{wc[k - 1], wd[k - 1]}, M{wc[k], wd[k]});
                wc[k] = r.c, wd[k] = r.d;
            }
        __syncthreads();
        if (wid) x = compose(M{wc[wid - 1], wd[wid - 1]}, x);
        auto apply = [](M q, uint64_t v) -> uint64_t {
            return q.c < 0 ? v + q.d : ((v + q.c + 7) & ~7ULL) + q.d;
        };
        const uint64_t end = apply(x, carry);
        // exclusive offset: the inclusive end of the previous block
        uint64_t prev = __shfl_up_sync(0xffffffffu, end, 1);
        if (lane == 0) prev = wid ? apply(M{wc[wid - 1], wd[wid - 1]}, carry) : carry;
        if (i < nb) boff[i] = prev;
        const uint64_t total = apply(M{wc[THREADS / 32 - 1], wd[THREADS / 32 - 1]}, carry);
        __syncthreads();
        carry = total;
    }
    if (threadIdx.x == 0) {
        fr.bits = (int64_t)carry;
        const int64_t zlen = 2 + (int64_t)((carry + 7) >> 3) + 4;
        fr.zlen = zlen;
        fr.nchunks = (zlen + IDAT - 1) / IDAT;
    }
}

__global__ void png_zero_kernel(Geo g, Work w, int n) {
    const int64_t gs = (int64_t)gridDim.x * blockDim.x;
    for (int f = 0; f < n; ++f) {
        const int64_t nw = (w.fr[f].bits + 31) >> 5;
        uint32_t *wd = w.words + (int64_t)f * g.wwords;
        for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nw; i += gs) wd[i] = 0;
    }
}

// LSB-first bit writer over a thread-exclusive bit range: the first and last words may be shared with neighbours
// (atomicOr), the words between are this thread's alone (plain stores onto the cleared buffer).
struct BitWriter {
    uint32_t *wd;
    int64_t widx, wfirst;
    uint64_t acc;
    int nacc;
    __device__ BitWriter(uint32_t *words, uint64_t pos)
        : wd(words), widx((int64_t)(pos >> 5)), wfirst((int64_t)(pos >> 5)), acc(0), nacc((int)(pos & 31)) {}
    __device__ __forceinline__ void put(uint64_t v, int len) {      // len <= 32
        acc |= v << nacc;
        nacc += len;
        if (nacc >= 32) {
            if (widx == wfirst) atomicOr(wd + widx, (uint32_t)acc);
            else wd[widx] = (uint32_t)acc;
            ++widx;
            acc >>= 32;
            nacc -= 32;
        }
    }
    __device__ __forceinline__ void flush() {
        if (nacc > 0) atomicOr(wd + widx, (uint32_t)acc);
    }
};

__global__ void __launch_bounds__(THREADS) png_emit_kernel(Geo g, Work w) {
    const int f = blockIdx.y;
    const int64_t b = blockIdx.x;
    const Frame &fr = w.fr[f];
    if (b >= fr.nblocks) return;
    const Plan &P = w.plan[(int64_t)f * g.maxb + b];
    const uint64_t pos = w.boff[(int64_t)f * g.maxb + b];
    const uint32_t last = b == fr.nblocks - 1;
    uint32_t *words = w.words + (int64_t)f * g.wwords;
    if (P.kind == 0) {
        const int64_t s0 = w.bstart[(int64_t)f * g.maxb + b], L = (int64_t)P.body_bits;
        if (threadIdx.x == 0) {
            BitWriter bw(words, pos);
            bw.put(last, 3);
            bw.flush();
        }
        const int64_t B = (int64_t)((pos + 3 + 7) >> 3);         // LEN, NLEN, then the bytes
        const uint8_t *F = w.F + (int64_t)f * g.Sp + s0;
        auto byte_at = [&](int64_t k) -> uint32_t {   // k-th byte from B
            if (k < 4) {
                const uint32_t len16 = (uint32_t)L & 0xffffu, v = len16 | ((~len16 & 0xffffu) << 16);
                return (v >> (8 * k)) & 0xffu;
            }
            return F[k - 4];
        };
        const int64_t total = 4 + L, w0 = B >> 2, w1 = (B + total + 3) >> 2;
        for (int64_t wi = w0 + threadIdx.x; wi < w1; wi += THREADS) {
            uint32_t v = 0;
            bool whole = true;
            for (int k = 0; k < 4; ++k) {
                const int64_t j = wi * 4 + k - B;
                if (j < 0 || j >= total) whole = false;
                else v |= byte_at(j) << (8 * k);
            }
            if (whole) words[wi] = v;
            else atomicOr(words + wi, v);
        }
        return;
    }
    __shared__ uint32_t code[L_CODES];
    for (int i = threadIdx.x; i < L_CODES; i += THREADS) code[i] = P.code[i];
    __syncthreads();
    const uint32_t dist = P.dist;
    const int dlen = (int)(dist >> 16);
    const int64_t a = b * BLOCK_SYMBOLS, e = min(a + BLOCK_SYMBOLS, fr.T);
    const uint16_t *syms = w.syms + (int64_t)f * g.S;
    constexpr int PER = (BLOCK_SYMBOLS + THREADS - 1) / THREADS;
    const int64_t i0 = a + (int64_t)threadIdx.x * PER, i1 = min(i0 + PER, e);
    auto sym_bits = [&](int sy) -> int {
        if (sy < 256) return (int)(code[sy] >> 16);
        const int lc = sy - 256, c = c_len.code[lc];
        return (int)(code[257 + c] >> 16) + c_extra_lbits[c] + dlen;
    };
    int64_t nbits = 0;
    for (int64_t i = i0; i < i1; ++i) nbits += sym_bits(syms[i]);
    if (threadIdx.x == THREADS - 1) nbits += code[END_BLOCK] >> 16;
    int64_t tot;
    const int64_t inc = cta_scan<int64_t>(nbits, 0, OpAdd(), &tot);
    const uint64_t data0 = pos + 3 + P.hdr_bits;
    if (threadIdx.x == 0) {
        BitWriter bw(words, pos);
        bw.put((P.kind << 1) | last, 3);
        for (uint32_t k = 0; k < P.hdr_bits; k += 32) {
            const int nb = (int)min(32u, P.hdr_bits - k);
            bw.put(nb == 32 ? P.hdr[k >> 5] : P.hdr[k >> 5] & ((1u << nb) - 1u), nb);
        }
        bw.flush();
    }
    if (nbits == 0) return;
    BitWriter bw(words, data0 + (uint64_t)(inc - nbits));
    for (int64_t i = i0; i < i1; ++i) {
        const int sy = syms[i];
        if (sy < 256) {
            bw.put(code[sy] & 0xffffu, (int)(code[sy] >> 16));
        } else {
            const int lc = sy - 256, c = c_len.code[lc];
            const uint32_t lcd = code[257 + c];
            const int xb = c_extra_lbits[c];
            uint64_t v = lcd & 0xffffu;
            int len = (int)(lcd >> 16);
            if (xb) {
                v |= (uint64_t)(lc - c_len.base[c]) << len;
                len += xb;
            }
            v |= (uint64_t)(dist & 0xffffu) << len;
            bw.put(v, len + dlen);
        }
    }
    if (threadIdx.x == THREADS - 1) bw.put(code[END_BLOCK] & 0xffffu, (int)(code[END_BLOCK] >> 16));
    bw.flush();
}

struct Header {
    uint8_t b[SIG_IHDR + 2];
};

__global__ void __launch_bounds__(THREADS) png_frame_kernel(Geo g, Work w, Header hdr, uint8_t *out, int64_t slot,
                                                            int64_t *lengths) {
    const int f = blockIdx.y;
    const int64_t c = blockIdx.x;
    const Frame &fr = w.fr[f];
    const int64_t nch = fr.nchunks, Z = fr.zlen, D = Z - 6;
    if (c >= nch) return;
    __shared__ uint32_t tab[256];
    __shared__ uint32_t crcs[THREADS], lens[THREADS];
    for (int i = threadIdx.x; i < 256; i += THREADS) tab[i] = c_crc.t[i];
    __syncthreads();
    uint8_t *dst = out + (int64_t)f * slot;
    const uint32_t a1 = (uint32_t)((1 + fr.s1) % ADLER_MOD), a2 = (uint32_t)(((uint64_t)g.S % ADLER_MOD + fr.s2) % ADLER_MOD);
    const uint32_t adler = (a2 << 16) | a1;
    const uint8_t *wb = reinterpret_cast<const uint8_t *>(w.words + (int64_t)f * g.wwords);
    const int64_t z0 = c * IDAT, plen = min((int64_t)IDAT, Z - z0);
    uint8_t *cd = dst + SIG_IHDR + c * (IDAT + 12);
    constexpr int SEG = IDAT / THREADS;
    uint32_t crc = 0xffffffffu;
    if (threadIdx.x == 0)
        for (int k = 0; k < 4; ++k) crc = tab[(crc ^ (uint8_t)"IDAT"[k]) & 0xff] ^ (crc >> 8);
    const int64_t k0 = (int64_t)threadIdx.x * SEG, k1 = min(k0 + SEG, plen);
    for (int64_t k = k0; k < k1; ++k) {
        const int64_t z = z0 + k;
        uint8_t v;
        if (z < 2) v = hdr.b[SIG_IHDR + z];
        else if (z < 2 + D) v = wb[z - 2];
        else v = (uint8_t)(adler >> (8 * (3 - (z - 2 - D))));
        cd[8 + k] = v;
        crc = tab[(crc ^ v) & 0xff] ^ (crc >> 8);
    }
    crcs[threadIdx.x] = ~crc;
    lens[threadIdx.x] = (uint32_t)max((int64_t)0, k1 - k0) + (threadIdx.x == 0 ? 4 : 0);
    __syncthreads();
    for (int d = 1; d < THREADS; d <<= 1) {
        if ((threadIdx.x & (2 * d - 1)) == 0) {
            crcs[threadIdx.x] = crc_combine(crcs[threadIdx.x], crcs[threadIdx.x + d], lens[threadIdx.x + d]);
            lens[threadIdx.x] += lens[threadIdx.x + d];
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        const uint32_t L = (uint32_t)plen, C = crcs[0];
        const uint8_t head[8] = {(uint8_t)(L >> 24), (uint8_t)(L >> 16), (uint8_t)(L >> 8), (uint8_t)L, 'I', 'D', 'A', 'T'};
        for (int k = 0; k < 8; ++k) cd[k] = head[k];
        for (int k = 0; k < 4; ++k) cd[8 + plen + k] = (uint8_t)(C >> (24 - 8 * k));
    }
    if (c == 0)
        for (int k = threadIdx.x; k < SIG_IHDR; k += THREADS) dst[k] = hdr.b[k];
    if (c == nch - 1 && threadIdx.x == 0) {
        uint8_t *e = cd + 12 + plen;
        const uint8_t iend[12] = {0, 0, 0, 0, 'I', 'E', 'N', 'D', 0xAE, 0x42, 0x60, 0x82};
        for (int k = 0; k < 12; ++k) e[k] = iend[k];
        lengths[f] = SIG_IHDR + nch * 12 + Z + 12;
    }
}

bool dims_ok(int H, int W) { return H >= 1 && H <= 65535 && W >= 1 && W <= 65535; }

}  // namespace

extern "C" int64_t avb_png_bound_bytes(int H, int W) {
    if (!dims_ok(H, W)) {
        avb::set_error("avb_png_bound_bytes: H and W must lie in [1, 65535]");
        return AVB_E_ARG;
    }
    const Geo g = geometry(H, W);
    // signature + IHDR, zlib stream (words, header, Adler-32), 12 framing bytes per IDAT, IEND
    return SIG_IHDR + g.wwords * 4 + 6 + 12 * g.maxchunks + 12;
}

extern "C" int64_t avb_png_workspace_bytes(int n, int H, int W) {
    if (!dims_ok(H, W) || n < 1 || n > 65535) {
        avb::set_error("avb_png_workspace_bytes: bad geometry");
        return AVB_E_ARG;
    }
    return carve(geometry(H, W), n, nullptr, nullptr);
}

extern "C" int avb_png_encode_u8(const uint8_t *in, int n, int H, int W, int64_t in_frame_stride, int64_t in_row_stride,
                                 const uint8_t *header_host, int header_len, uint8_t *out, int64_t out_slot_stride,
                                 int64_t *out_lengths_dev, void *workspace_dev, avb_stream_t stream) {
    AVB_REQUIRE(in && header_host && out && out_lengths_dev && workspace_dev, "null pointer");
    AVB_REQUIRE(n >= 1 && n <= 65535 && dims_ok(H, W), "n must lie in [1, 65535], H and W in [1, 65535]");
    AVB_REQUIRE(in_row_stride >= 3LL * W && (n == 1 || in_frame_stride >= in_row_stride * (H - 1) + 3LL * W),
                "input strides overlap");
    AVB_REQUIRE(header_len == AVB_PNG_HEADER_LEN, "header_len must be AVB_PNG_HEADER_LEN (signature, IHDR, CMF/FLG)");
    AVB_REQUIRE(out_slot_stride >= avb_png_bound_bytes(H, W), "output slot smaller than avb_png_bound_bytes(H, W)");
    AVB_REQUIRE(((uintptr_t)workspace_dev & 15) == 0, "workspace must be 16-byte aligned");
    const Geo g = geometry(H, W);
    Header hdr;
    memcpy(hdr.b, header_host, header_len);
    Work w;
    carve(g, n, (uint8_t *)workspace_dev, &w);
    cudaStream_t st = (cudaStream_t)stream;
    const dim3 tiles((unsigned)g.ntiles, n), blocks((unsigned)(g.maxb - 1), n);
    AVB_CUDA_OK(cudaMemsetAsync(w.fr, 0, n * sizeof(Frame), st));
    {
        AVB_TIMED("png_filter", st);
        png_filter_kernel<<<tiles, THREADS, 0, st>>>(in, in_frame_stride, in_row_stride, g, w);
    }
    {
        AVB_TIMED("png_run_carry", st);
        png_run_carry_kernel<<<n, THREADS, 0, st>>>(g, w);
    }
    {
        AVB_TIMED("png_symbols_count", st);
        png_symbols_kernel<false><<<tiles, THREADS, 0, st>>>(g, w);
    }
    {
        AVB_TIMED("png_sym_scan", st);
        png_sym_scan_kernel<<<n, THREADS, 0, st>>>(g, w);
    }
    {
        AVB_TIMED("png_symbols_write", st);
        png_symbols_kernel<true><<<tiles, THREADS, 0, st>>>(g, w);
    }
    {
        AVB_TIMED("png_block_plan", st);
        png_block_plan_kernel<<<blocks, THREADS, 0, st>>>(g, w);
    }
    {
        AVB_TIMED("png_block_scan", st);
        png_block_scan_kernel<<<n, THREADS, 0, st>>>(g, w);
    }
    {
        AVB_TIMED("png_zero", st);
        png_zero_kernel<<<avb::sm_count() * 4, 256, 0, st>>>(g, w, n);
    }
    {
        AVB_TIMED("png_emit", st);
        png_emit_kernel<<<blocks, THREADS, 0, st>>>(g, w);
    }
    {
        AVB_TIMED("png_frame", st);
        png_frame_kernel<<<dim3((unsigned)g.maxchunks, n), THREADS, 0, st>>>(g, w, hdr, out, out_slot_stride,
                                                                            out_lengths_dev);
    }
    AVB_CUDA_OK(cudaGetLastError());
    return AVB_OK;
}
