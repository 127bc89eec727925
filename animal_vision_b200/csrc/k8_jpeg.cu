// K8 -- batched baseline JPEG encoder, byte-identical to cv2.imencode(".jpg") with OpenCV's defaults
// (libjpeg-turbo: 4:2:0, standard Huffman tables, no restart interval).  Every stage is integer arithmetic, so
// the device restates libjpeg bit for bit (oracle/jpeg.py is the NumPy statement of the same stages):
//   jpeg_transform  one CTA per strip of 8 MCUs (16 x 128 px): BGR (or RGB) gather with edge replication, jccolor.c
//                   fixed-point YCbCr, jcsample.c h2v2 (bias 1, 2), jfdctint.c islow, jcdctmgr.c quantisation,
//                   jccoefct.c dummy blocks; writes zigzag int16 coefficients, quantised DCs and per-block
//                   code lengths (the DC code of blocks 0 / Cb / Cr waits for the previous MCU's DCs)
//   jpeg_mcu_scan   one CTA per frame: MCU lengths (+ the cross-MCU DC codes, a neighbour read) -> 64-bit
//                   exclusive bit offsets, total bits
//   jpeg_zero       clears exactly the words the frame's bits occupy; the 1-bits padding the last byte go in here
//   jpeg_emit       one thread per 8x8 block writes its Huffman bits at its offset (atomicOr on the word buffer)
//   jpeg_ff_count   0xFF bytes per 16-byte chunk
//   jpeg_ff_scan    one CTA per frame: chunk offsets of the stuffed stream, header + EOI, total length
//   jpeg_stuff      scatter of the bytes with 0x00 after every 0xFF (jchuff.c emit_byte)
// The optimized mode (avb_jpeg_opt_encode_u8, cv2.IMWRITE_JPEG_OPTIMIZE) codes each frame with Huffman tables built from
// its own symbol counts.  The template flag OPT of the shared kernels selects it; the standard instances are unchanged.
//   jpeg_transform  counts the AC symbols of its blocks in shared memory, adds them to the frame's 64-bit counters;
//                   writes no code lengths (the tables are not known yet)
//   jpeg_dc_hist    one thread per MCU: DC symbol counts (they need the previous MCU's DCs)
//   jpeg_tables     one CTA per frame, one warp per table: jchuff.c jpeg_gen_optimal_table, jpeg_make_c_derived_tbl and
//                   the DHT segment
//   jpeg_blen       one thread per block: its code length from the frame's tables
// then jpeg_mcu_scan and jpeg_emit read the frame's tables from shared memory, jpeg_ff_scan writes the header prefix,
// the frame's four DHT segments and the SOS segment, and jpeg_stuff starts the data after that frame's header.
#include <string.h>

#include "avb_common.cuh"

namespace {

constexpr int STRIP = 8;                       // MCUs per transform CTA
constexpr int TF_THREADS = STRIP * 6 * 8;      // 8 threads per 8x8 block
constexpr int SCAN_THREADS = 512, SCAN_ITEMS = 8;
constexpr int CHUNK = 16;                      // bytes per 0xFF-stuffing chunk
// Each of the 64 coefficients of a block codes to at most a 16-bit Huffman code plus 11 magnitude bits (a ZRL
// replaces 16 zero coefficients with one code and an EOB one or more zeros), so one MCU of six blocks needs at most
// 6 * 64 * 27 bits = 1296 bytes of entropy-coded data before 0xFF stuffing.
constexpr int64_t MCU_BYTES_MAX = 6 * 64 * 27 / 8;

struct HuffSpec {
    uint8_t bits[16];
    uint8_t vals[162];
};
// ITU-T T.81 Annex K.3, as jcparam.c / jstdhuff.c install them
constexpr HuffSpec DC_L = {{0, 1, 5, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0, 0, 0}, {0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11}};
constexpr HuffSpec DC_C = {{0, 3, 1, 1, 1, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0}, {0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11}};
constexpr HuffSpec AC_L = {{0, 2, 1, 3, 3, 2, 4, 3, 5, 5, 4, 4, 0, 0, 1, 125},
    {1, 2, 3, 0, 4, 17, 5, 18, 33, 49, 65, 6, 19, 81, 97, 7, 34, 113, 20, 50, 129, 145, 161, 8, 35, 66, 177, 193, 21, 82,
     209, 240, 36, 51, 98, 114, 130, 9, 10, 22, 23, 24, 25, 26, 37, 38, 39, 40, 41, 42, 52, 53, 54, 55, 56, 57, 58, 67, 68,
     69, 70, 71, 72, 73, 74, 83, 84, 85, 86, 87, 88, 89, 90, 99, 100, 101, 102, 103, 104, 105, 106, 115, 116, 117, 118, 119,
     120, 121, 122, 131, 132, 133, 134, 135, 136, 137, 138, 146, 147, 148, 149, 150, 151, 152, 153, 154, 162, 163, 164, 165,
     166, 167, 168, 169, 170, 178, 179, 180, 181, 182, 183, 184, 185, 186, 194, 195, 196, 197, 198, 199, 200, 201, 202, 210,
     211, 212, 213, 214, 215, 216, 217, 218, 225, 226, 227, 228, 229, 230, 231, 232, 233, 234, 241, 242, 243, 244, 245, 246,
     247, 248, 249, 250}};
constexpr HuffSpec AC_C = {{0, 2, 1, 2, 4, 4, 3, 4, 7, 5, 4, 4, 0, 1, 2, 119},
    {0, 1, 2, 3, 17, 4, 5, 33, 49, 6, 18, 65, 81, 7, 97, 113, 19, 34, 50, 129, 8, 20, 66, 145, 161, 177, 193, 9, 35, 51, 82,
     240, 21, 98, 114, 209, 10, 22, 36, 52, 225, 37, 241, 23, 24, 25, 26, 38, 39, 40, 41, 42, 53, 54, 55, 56, 57, 58, 67, 68,
     69, 70, 71, 72, 73, 74, 83, 84, 85, 86, 87, 88, 89, 90, 99, 100, 101, 102, 103, 104, 105, 106, 115, 116, 117, 118, 119,
     120, 121, 122, 130, 131, 132, 133, 134, 135, 136, 137, 138, 146, 147, 148, 149, 150, 151, 152, 153, 154, 162, 163, 164,
     165, 166, 167, 168, 169, 170, 178, 179, 180, 181, 182, 183, 184, 185, 186, 194, 195, 196, 197, 198, 199, 200, 201, 202,
     210, 211, 212, 213, 214, 215, 216, 217, 218, 226, 227, 228, 229, 230, 231, 232, 233, 234, 242, 243, 244, 245, 246, 247,
     248, 249, 250}};

// (length << 16) | code of every symbol; [0] luma, [1] chroma
struct HuffTabs {
    uint32_t dc[2][16];
    uint32_t ac[2][256];
};

constexpr void derive(const HuffSpec &s, uint32_t *out) {     // jchuff.c jpeg_make_c_derived_tbl
    int code = 0, k = 0;
    for (int L = 1; L <= 16; ++L) {
        for (int i = 0; i < s.bits[L - 1]; ++i) out[s.vals[k++]] = ((uint32_t)L << 16) | (uint32_t)code++;
        code <<= 1;
    }
}

constexpr HuffTabs make_huff() {
    HuffTabs t{};
    derive(DC_L, t.dc[0]);
    derive(DC_C, t.dc[1]);
    derive(AC_L, t.ac[0]);
    derive(AC_C, t.ac[1]);
    return t;
}

__constant__ HuffTabs c_huff = make_huff();

// The codes a kernel reads: the standard tables in constant memory, or (OPT) the frame's own in shared memory
template <bool OPT>
struct Codes {
    const uint32_t (*dct)[16];
    const uint32_t (*act)[256];
    __device__ __forceinline__ uint32_t dc(int tab, int s) const {
        if constexpr (OPT) return dct[tab][s];
        else return c_huff.dc[tab][s];
    }
    __device__ __forceinline__ uint32_t ac(int tab, int sym) const {
        if constexpr (OPT) return act[tab][sym];
        else return c_huff.ac[tab][sym];
    }
};

// natural index -> zigzag position
__constant__ uint8_t c_izz[64] = {0,  1,  5,  6,  14, 15, 27, 28, 2,  4,  7,  13, 16, 26, 29, 42, 3,  8,  12, 17, 25, 30,
                                  41, 43, 9,  11, 18, 24, 31, 40, 44, 53, 10, 19, 23, 32, 39, 45, 52, 54, 20, 22, 33, 38,
                                  46, 51, 55, 60, 21, 34, 37, 47, 50, 56, 59, 61, 35, 36, 48, 49, 57, 58, 62, 63};

struct QDiv {
    uint16_t d[2][64];          // 8 * quantiser in natural order (the islow output is scaled by 8); [0] luma, [1] chroma
};

struct Header {
    uint8_t b[AVB_JPEG_HEADER_MAX];
};

// A DHT segment: marker, length, class / id, bits[1..16], up to 256 values
constexpr int DHT_SEG_MAX = 4 + 1 + 16 + 256;
constexpr int DHT_BYTES = (4 * DHT_SEG_MAX + 15) & ~15;     // the four segments of a frame
// What the four segments take at most: an 8-bit baseline DC table holds the sizes 0..11, an AC table the 160 (run, size)
// symbols with sizes 1..10, ZRL and EOB -- the symbol sets of the standard tables (jchuff.c MAX_COEF_BITS)
constexpr int DHT_LEN_MAX = 2 * (4 + 1 + 16 + 12) + 2 * (4 + 1 + 16 + 162);

struct Geo {
    int H, W, mw, mh, bw, bh;
    int64_t M;                  // MCUs per frame
    int64_t wbytes;             // entropy word buffer bytes per frame
    int64_t chunks;             // stuffing chunks per frame
};

Geo geometry(int H, int W) {
    Geo g;
    g.H = H;
    g.W = W;
    g.mw = (W + 15) / 16;
    g.mh = (H + 15) / 16;
    g.bw = (W + 7) / 8;
    g.bh = (H + 7) / 8;
    g.M = (int64_t)g.mw * g.mh;
    g.wbytes = g.M * MCU_BYTES_MAX;     // a multiple of 16
    g.chunks = g.wbytes / CHUNK;
    return g;
}

// workspace carve-up; every part 16-byte aligned
struct Work {
    int16_t *coef;              // [n][M][6][64] zigzag
    uint16_t *blen;             // [n][M][8] bits per block (blocks 0, 4, 5 without their DC code)
    int16_t *dcs;               // [n][M][8] quantised DC per block
    uint64_t *off;              // [n][M] bit offset of each MCU
    uint32_t *words;            // [n][wbytes / 4] entropy bits, MSB first
    uint32_t *ffcnt;            // [n][chunks] 0xFF bytes per chunk, then (in place) their exclusive prefix
    uint64_t *bits;             // [n] total entropy bits
};

// the optimized mode's part of the workspace, after carve's
struct Opt {
    uint64_t *freq;             // [n][4][256] symbol counts: DC0, AC0, DC1, AC1
    HuffTabs *tabs;             // [n] the frame's codes
    uint8_t *dht;               // [n][DHT_BYTES] the frame's DHT segments, back to back
    int *dhtlen;                // [n] their bytes
    int *hlen;                  // [n] header bytes (prefix + DHT segments + SOS)
    int slen;                   // SOS bytes; the header prefix's are the kernels' hlen argument
};

int64_t carve(const Geo &g, int n, uint8_t *base, Work *w) {
    int64_t o = 0;
    auto take = [&](int64_t bytes) {
        uint8_t *p = base ? base + o : nullptr;
        o += (bytes + 15) & ~(int64_t)15;
        return p;
    };
    const int64_t nm = (int64_t)n * g.M;
    Work t;
    t.coef = (int16_t *)take(nm * 384 * 2);
    t.blen = (uint16_t *)take(nm * 16);
    t.dcs = (int16_t *)take(nm * 16);
    t.off = (uint64_t *)take(nm * 8);
    t.words = (uint32_t *)take((int64_t)n * g.wbytes);
    t.ffcnt = (uint32_t *)take((int64_t)n * g.chunks * 4);
    t.bits = (uint64_t *)take((int64_t)n * 8);
    if (w) *w = t;
    return o;
}

int64_t carve_opt(const Geo &g, int n, uint8_t *base, Opt *op) {
    int64_t o = carve(g, n, nullptr, nullptr);
    auto take = [&](int64_t bytes) {
        uint8_t *p = base ? base + o : nullptr;
        o += (bytes + 15) & ~(int64_t)15;
        return p;
    };
    Opt t{};
    t.freq = (uint64_t *)take((int64_t)n * 4 * 256 * 8);
    t.tabs = (HuffTabs *)take((int64_t)n * sizeof(HuffTabs));
    t.dht = take((int64_t)n * DHT_BYTES);
    t.dhtlen = (int *)take((int64_t)n * 4);
    t.hlen = (int *)take((int64_t)n * 4);
    if (op) *op = t;
    return o;
}

__device__ __forceinline__ int nbits_of(int v) {
    v = abs(v);
    return v ? 32 - __clz(v) : 0;
}

template <bool OPT>
__device__ __forceinline__ int dc_len(const Codes<OPT> &c, int tab, int diff) {
    const int s = nbits_of(diff);
    return (int)(c.dc(tab, s) >> 16) + s;
}

__device__ __forceinline__ int descale(int x, int n) { return (x + (1 << (n - 1))) >> n; }

// jfdctint.c jpeg_fdct_islow, one row (first pass) or one column (second pass)
template <bool SECOND>
__device__ __forceinline__ void fdct8(const int *d, int *o) {
    constexpr int SH = SECOND ? 13 + 2 : 13 - 2;
    const int tmp0 = d[0] + d[7], tmp7 = d[0] - d[7], tmp1 = d[1] + d[6], tmp6 = d[1] - d[6];
    const int tmp2 = d[2] + d[5], tmp5 = d[2] - d[5], tmp3 = d[3] + d[4], tmp4 = d[3] - d[4];
    const int tmp10 = tmp0 + tmp3, tmp13 = tmp0 - tmp3, tmp11 = tmp1 + tmp2, tmp12 = tmp1 - tmp2;
    o[0] = SECOND ? descale(tmp10 + tmp11, 2) : (tmp10 + tmp11) * 4;
    o[4] = SECOND ? descale(tmp10 - tmp11, 2) : (tmp10 - tmp11) * 4;
    int z1 = (tmp12 + tmp13) * 4433;
    o[2] = descale(z1 + tmp13 * 6270, SH);
    o[6] = descale(z1 - tmp12 * 15137, SH);
    z1 = tmp4 + tmp7;
    int z2 = tmp5 + tmp6, z3 = tmp4 + tmp6, z4 = tmp5 + tmp7;
    const int z5 = (z3 + z4) * 9633;
    const int t4 = tmp4 * 2446, t5 = tmp5 * 16819, t6 = tmp6 * 25172, t7 = tmp7 * 12299;
    z1 *= -7373;
    z2 *= -20995;
    z3 = z3 * -16069 + z5;
    z4 = z4 * -3196 + z5;
    o[7] = descale(t4 + z1 + z3, SH);
    o[5] = descale(t5 + z2 + z4, SH);
    o[3] = descale(t6 + z2 + z3, SH);
    o[1] = descale(t7 + z1 + z4, SH);
}

// RGB: the frames hold R, G, B (avb_jpeg_encode_rgb_u8); everything after the gather is shared
// OPT: AC symbol counts instead of code lengths
template <bool RGB, bool OPT>
__global__ void __launch_bounds__(TF_THREADS) jpeg_transform_kernel(const uint8_t *__restrict__ in, int64_t fs, int64_t rs,
                                                                     Geo g, QDiv qd, Work w, Opt op) {
    __shared__ uint8_t sY[16][128], sCb[16][128], sCr[16][128], sC[2][8][64];
    __shared__ int work[STRIP * 6][8][9];
    __shared__ __align__(16) int16_t qz[STRIP * 6][64];
    __shared__ uint16_t sdiv[2][64];
    __shared__ uint8_t sizz[64];
    const int tid = threadIdx.x, f = blockIdx.z, my = blockIdx.y, mx0 = blockIdx.x * STRIP;
    uint32_t *hist = nullptr;                                   // [2][256] AC counts of the CTA: luma, chroma
    if constexpr (OPT) {
        __shared__ uint32_t shist[2 * 256];
        hist = shist;
        for (int i = tid; i < 2 * 256; i += TF_THREADS) hist[i] = 0;
    }
    if (tid < 128) sdiv[tid >> 6][tid & 63] = qd.d[tid >> 6][tid & 63];
    if (tid < 64) sizz[tid] = c_izz[tid];
    const uint8_t *fin = in + (int64_t)f * fs;
    for (int p = tid; p < 16 * 128; p += TF_THREADS) {          // columns / rows past the edge repeat the last one
        const int r = p >> 7, c = p & 127;
        const int gy = min(my * 16 + r, g.H - 1), gx = min(mx0 * 16 + c, g.W - 1);
        const uint8_t *px = fin + gy * rs + gx * 3;
        const int b = px[RGB ? 2 : 0], gg = px[1], rr = px[RGB ? 0 : 2];
        sY[r][c] = (uint8_t)((19595 * rr + 38470 * gg + 7471 * b + 32768) >> 16);
        sCb[r][c] = (uint8_t)((-11059 * rr - 21709 * gg + 32768 * b + (128 << 16) + 32767) >> 16);
        sCr[r][c] = (uint8_t)((32768 * rr - 27439 * gg - 5329 * b + (128 << 16) + 32767) >> 16);
    }
    __syncthreads();
    const int ch = (g.H + 1) >> 1;
    for (int p = tid; p < 2 * 8 * 64; p += TF_THREADS) {        // h2v2; downsampled rows below the image repeat the last
        const int pl = p >> 9, k = (p >> 6) & 7, x = p & 63;
        const int r0 = 2 * (min(my * 8 + k, ch - 1) - my * 8), c0 = 2 * x;
        const uint8_t(*P)[128] = pl ? sCr : sCb;
        const int s = P[r0][c0] + P[r0][c0 + 1] + P[r0 + 1][c0] + P[r0 + 1][c0 + 1];
        sC[pl][k][x] = (uint8_t)((s + 1 + (x & 1)) >> 2);
    }
    __syncthreads();
    const int bl = tid >> 3, lane = tid & 7, j = bl / 6, b = bl - j * 6, mx = mx0 + j;
    const bool right = (g.bw & 1) && mx == g.mw - 1, bottom = (g.bh & 1) && my == g.mh - 1;
    const bool dummy = (right && (b == 1 || b == 3)) || (bottom && (b == 2 || b == 3));     // luma blocks only
    {
        int d[8], o[8];
#pragma unroll
        for (int c = 0; c < 8; ++c) {
            int v;
            if (b < 4) v = sY[(b >> 1) * 8 + lane][j * 16 + (b & 1) * 8 + c];
            else v = sC[b - 4][lane][j * 8 + c];
            d[c] = v - 128;
        }
        fdct8<false>(d, o);
#pragma unroll
        for (int c = 0; c < 8; ++c) work[bl][lane][c] = o[c];
    }
    __syncthreads();
    {
        int d[8], o[8];
#pragma unroll
        for (int r = 0; r < 8; ++r) d[r] = work[bl][r][lane];
        fdct8<true>(d, o);
        const int tab = b >= 4;
#pragma unroll
        for (int r = 0; r < 8; ++r) {
            const int nat = r * 8 + lane, div = sdiv[tab][nat];
            const int v = o[r], mag = (abs(v) + (div >> 1)) / div;
            qz[bl][sizz[nat]] = dummy ? 0 : (int16_t)(v < 0 ? -mag : mag);
        }
    }
    __syncthreads();
    if (tid < STRIP) {                // dummy blocks take the DC of the preceding block (jccoefct.c compress_data)
        const int m0 = tid * 6, mxt = mx0 + tid;
        const bool rt = (g.bw & 1) && mxt == g.mw - 1;
        if (rt) {
            qz[m0 + 1][0] = qz[m0][0];
            qz[m0 + 3][0] = qz[m0 + 2][0];
        }
        if (bottom) {
            qz[m0 + 2][0] = qz[m0 + 1][0];
            qz[m0 + 3][0] = qz[m0 + 1][0];
        }
    }
    __syncthreads();
    const int na = min(STRIP, g.mw - mx0);
    const int64_t mcu0 = (int64_t)f * g.M + (int64_t)my * g.mw + mx0;
    if (tid < na * 48) reinterpret_cast<int4 *>(w.coef + mcu0 * 384)[tid] = reinterpret_cast<const int4 *>(&qz[0][0])[tid];
    // code length of the block: every nonzero AC coefficient's run follows from the nonzero mask alone
    uint64_t mask = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) mask |= (uint64_t)(qz[bl][lane * 8 + k] != 0) << (lane * 8 + k);
    mask |= __shfl_xor_sync(0xffffffffu, mask, 1);
    mask |= __shfl_xor_sync(0xffffffffu, mask, 2);
    mask |= __shfl_xor_sync(0xffffffffu, mask, 4);
    mask &= ~1ull;
    const int tab = b >= 4;
    if constexpr (OPT) {              // jchuff.c htest_one_block; blocks of MCUs past the right edge are not coded
        if (j < na) {
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                const int zz = lane * 8 + k;
                if ((mask >> zz) & 1) {
                    const uint64_t below = mask & ((1ull << zz) - 1);
                    const int prev = below ? 63 - __clzll((long long)below) : 0;
                    const int run = zz - prev - 1;
                    if (run >= 16) atomicAdd(&hist[tab * 256 + 0xF0], (uint32_t)(run >> 4));
                    atomicAdd(&hist[tab * 256 + (((run & 15) << 4) | nbits_of(qz[bl][zz]))], 1u);
                }
            }
            if (lane == 0) {
                if (!(mask >> 63)) atomicAdd(&hist[tab * 256], 1u);
                w.dcs[(mcu0 + j) * 8 + b] = qz[bl][0];
            }
        }
        __syncthreads();
        for (int i = tid; i < 2 * 256; i += TF_THREADS)
            if (hist[i])
                atomicAdd((unsigned long long *)&op.freq[((int64_t)f * 4 + 2 * (i >> 8) + 1) * 256 + (i & 255)],
                          (unsigned long long)hist[i]);
        return;
    }
    const int zrl = (int)(c_huff.ac[tab][0xF0] >> 16);
    int len = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        const int zz = lane * 8 + k;
        if ((mask >> zz) & 1) {
            const uint64_t below = mask & ((1ull << zz) - 1);
            const int prev = below ? 63 - __clzll((long long)below) : 0;
            const int run = zz - prev - 1, s = nbits_of(qz[bl][zz]);
            len += (run >> 4) * zrl + (int)(c_huff.ac[tab][((run & 15) << 4) | s] >> 16) + s;
        }
    }
    if (lane == 0) {
        if (!(mask >> 63)) len += (int)(c_huff.ac[tab][0] >> 16);
        if (b >= 1 && b <= 3) len += dc_len(Codes<false>{}, 0, qz[bl][0] - qz[bl - 1][0]);
    }
    len += __shfl_xor_sync(0xffffffffu, len, 1);
    len += __shfl_xor_sync(0xffffffffu, len, 2);
    len += __shfl_xor_sync(0xffffffffu, len, 4);
    if (lane == 0 && j < na) {
        w.blen[(mcu0 + j) * 8 + b] = (uint16_t)len;
        w.dcs[(mcu0 + j) * 8 + b] = qz[bl][0];
    }
}

// Exclusive scan of n items over one CTA of SCAN_THREADS threads, SCAN_ITEMS consecutive items per thread and tile.
// item(i) -> uint64_t, out(i, prefix).  Returns the total.
template <class Item, class Out>
__device__ uint64_t block_scan(int64_t n, Item item, Out out) {
    constexpr int NW = SCAN_THREADS / 32;
    __shared__ uint64_t wtot[NW];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    uint64_t carry = 0;
    for (int64_t base = 0; base < n; base += (int64_t)SCAN_THREADS * SCAN_ITEMS) {
        const int64_t i0 = base + (int64_t)threadIdx.x * SCAN_ITEMS;
        uint64_t v[SCAN_ITEMS], s = 0;
#pragma unroll
        for (int k = 0; k < SCAN_ITEMS; ++k) {
            v[k] = i0 + k < n ? item(i0 + k) : 0;
            s += v[k];
        }
        uint64_t x = s;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint64_t y = __shfl_up_sync(0xffffffffu, x, o);
            if (lane >= o) x += y;
        }
        if (lane == 31) wtot[wid] = x;
        __syncthreads();
        if (wid == 0) {
            uint64_t t = lane < NW ? wtot[lane] : 0;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint64_t y = __shfl_up_sync(0xffffffffu, t, o);
                if (lane >= o) t += y;
            }
            if (lane < NW) wtot[lane] = t;
        }
        __syncthreads();
        uint64_t e = carry + (wid ? wtot[wid - 1] : 0) + x - s;
#pragma unroll
        for (int k = 0; k < SCAN_ITEMS; ++k) {
            if (i0 + k < n) out(i0 + k, e);
            e += v[k];
        }
        carry += wtot[NW - 1];
        __syncthreads();
    }
    return carry;
}

struct Dc8 {
    int v[8];
};
__device__ __forceinline__ Dc8 load_dc(const int16_t *p) {
    const int4 q = *reinterpret_cast<const int4 *>(p);
    const int u[4] = {q.x, q.y, q.z, q.w};
    Dc8 d;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        d.v[2 * k] = (int)(int16_t)(u[k] & 0xffff);
        d.v[2 * k + 1] = u[k] >> 16;
    }
    return d;
}

// the DC codes that need the previous MCU: block 0 after the previous Y11, Cb and Cr after theirs
template <bool OPT>
__device__ __forceinline__ int cross_dc_len(const Codes<OPT> &c, const Dc8 &d, const Dc8 &p) {
    return dc_len(c, 0, d.v[0] - p.v[3]) + dc_len(c, 1, d.v[4] - p.v[4]) + dc_len(c, 1, d.v[5] - p.v[5]);
}

__device__ __forceinline__ Dc8 prev_dc(const int16_t *dcs, int64_t fm, int64_t m) {
    if (m > 0) return load_dc(dcs + (fm - 1) * 8);
    Dc8 z;
#pragma unroll
    for (int k = 0; k < 8; ++k) z.v[k] = 0;
    return z;
}

// The frame's codes into shared memory (OPT); every thread of the CTA takes part
__device__ __forceinline__ void load_tabs(HuffTabs *s, const HuffTabs *t) {
    static_assert(sizeof(HuffTabs) % 16 == 0, "HuffTabs is copied in 16-byte pieces");
    for (int i = threadIdx.x; i < (int)(sizeof(HuffTabs) / 16); i += blockDim.x)
        reinterpret_cast<uint4 *>(s)[i] = reinterpret_cast<const uint4 *>(t)[i];
    __syncthreads();
}

// DC symbol counts of every block (OPT)
__global__ void __launch_bounds__(256) jpeg_dc_hist_kernel(Geo g, Work w, Opt op) {
    __shared__ uint32_t hist[2][16];                // luma, chroma; a DC size is at most 12
    const int f = blockIdx.y;
    const int64_t m = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (threadIdx.x < 32) hist[threadIdx.x >> 4][threadIdx.x & 15] = 0;
    __syncthreads();
    if (m < g.M) {
        const int64_t fm = (int64_t)f * g.M + m;
        const Dc8 d = load_dc(w.dcs + fm * 8), p = prev_dc(w.dcs, fm, m);
#pragma unroll
        for (int k = 0; k < 6; ++k) {               // predictors as jpeg_emit's
            const int pk = k == 0 ? p.v[3] : (k < 4 ? d.v[k - 1] : p.v[k]);
            atomicAdd(&hist[k >= 4][nbits_of(d.v[k] - pk)], 1u);
        }
    }
    __syncthreads();
    if (threadIdx.x < 32) {
        const uint32_t v = hist[threadIdx.x >> 4][threadIdx.x & 15];
        if (v)
            atomicAdd((unsigned long long *)&op.freq[((int64_t)f * 4 + 2 * (threadIdx.x >> 4)) * 256 + (threadIdx.x & 15)],
                      (unsigned long long)v);
    }
}

// One CTA per frame, one warp per table t (DC0, AC0, DC1, AC1).  jchuff.c jpeg_gen_optimal_table: symbol 256 with count 1
// reserves the all-ones code; each step merges the two least frequent trees c1, c2 (the smallest count, ties to the
// largest symbol, counts above libjpeg's initial v = 10^9 never taken) and lengthens the codes of both.  The symbols with
// a nonzero count are exactly the roots of the trees, so a tree is kept as a label (its root) on each symbol.  Then the
// lengths above 16 are folded down, the values are ordered by (unlimited) code length, then symbol, and take canonical
// codes (jpeg_make_c_derived_tbl); the warp writes the frame's codes and its DHT segment.
__global__ void __launch_bounds__(128) jpeg_tables_kernel(Opt op) {
    constexpr int K = 9;                            // symbols per lane: lane + 32 k covers 0..256
    constexpr uint64_t V0 = 1000000000ull, NONE = ~0ull;
    __shared__ int sbits[4][33], sstart[4][33], sfirst[4][17], scode[4][17], snsym[4];
    __shared__ uint8_t sval[4][256];
    const int f = blockIdx.x, t = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint64_t *fr = op.freq + ((int64_t)f * 4 + t) * 256;
    uint64_t fq[K];
    int cs[K], lab[K];
#pragma unroll
    for (int k = 0; k < K; ++k) {
        const int i = lane + 32 * k;
        fq[k] = i < 256 ? fr[i] : (uint64_t)(i == 256);
        cs[k] = 0;
        lab[k] = i;
    }
    for (int i = lane; i < 33; i += 32) sbits[t][i] = sstart[t][i] = 0;
    // the least key (count << 9) | (256 - symbol) among the candidates: the smallest count, ties to the largest symbol
    auto least = [&](int skip) {
        uint64_t m = NONE;
#pragma unroll
        for (int k = 0; k < K; ++k) {
            const int i = lane + 32 * k;
            if (fq[k] && fq[k] <= V0 && i != skip) m = min(m, (fq[k] << 9) | (uint64_t)(256 - i));
        }
#pragma unroll
        for (int o = 16; o; o >>= 1) m = min(m, __shfl_xor_sync(0xffffffffu, m, o));
        return m;
    };
    for (;;) {
        const uint64_t k1 = least(-1);
        const int c1 = 256 - (int)(k1 & 511);
        const uint64_t k2 = k1 == NONE ? NONE : least(c1);
        if (k2 == NONE) break;
        const int c2 = 256 - (int)(k2 & 511);
#pragma unroll
        for (int k = 0; k < K; ++k) {
            const int i = lane + 32 * k;
            if (lab[k] == c1 || lab[k] == c2) {
                ++cs[k];
                lab[k] = c1;
            }
            if (i == c1) fq[k] += k2 >> 9;
            if (i == c2) fq[k] = 0;
        }
    }
    __syncwarp();
#pragma unroll
    for (int k = 0; k < K; ++k) {                   // jpeg_gen_optimal_table allows code lengths up to 32
        const int i = lane + 32 * k;
        if (cs[k] && i <= 256) {
            atomicAdd(&sbits[t][min(cs[k], 32)], 1);
            if (i < 256) atomicAdd(&sstart[t][min(cs[k], 32)], 1);
        }
    }
    __syncwarp();
    if (lane == 0) {
        int *bits = sbits[t];
        for (int i = 32; i > 16; --i)
            while (bits[i] > 0) {
                int j = i - 2;
                while (bits[j] == 0) --j;
                bits[i] -= 2;
                bits[i - 1] += 1;
                bits[j + 1] += 2;
                bits[j] -= 1;
            }
        int i = 16;
        while (bits[i] == 0) --i;
        bits[i] -= 1;                               // the reserved code
        int s = 0;
        for (int L = 1; L <= 32; ++L) {             // first value position of each unlimited length
            const int c = sstart[t][L];
            sstart[t][L] = s;
            s += c;
        }
        int code = 0, p = 0;
        for (int L = 1; L <= 16; ++L) {             // canonical codes: first position and first code of each length
            sfirst[t][L] = p;
            scode[t][L] = code;
            p += bits[L];
            code = (code + bits[L]) << 1;
        }
        snsym[t] = p;
    }
    __syncwarp();
    int pos[K];
#pragma unroll
    for (int k = 0; k < K; ++k) {                   // value positions, symbols of one length in increasing order
        const int i = lane + 32 * k;
        const int L = i < 256 && cs[k] ? min(cs[k], 32) : 0;
        const unsigned same = __match_any_sync(0xffffffffu, L);
        pos[k] = L ? sstart[t][L] + __popc(same & ((1u << lane) - 1u)) : -1;
        __syncwarp();
        if (L && lane == __ffs(same) - 1) sstart[t][L] += __popc(same);
        __syncwarp();
    }
    HuffTabs *tabs = op.tabs + f;
    uint32_t *dst = t & 1 ? tabs->ac[t >> 1] : tabs->dc[t >> 1];
    const int nent = t & 1 ? 256 : 16;
#pragma unroll
    for (int k = 0; k < K; ++k) {
        const int i = lane + 32 * k, p = pos[k];
        if (p >= 0) sval[t][p] = (uint8_t)i;
        if (i < nent) {
            uint32_t e = 0;
            if (p >= 0)
                for (int L = 1; L <= 16; ++L)
                    if (p >= sfirst[t][L] && p < sfirst[t][L] + sbits[t][L])
                        e = ((uint32_t)L << 16) | (uint32_t)(scode[t][L] + p - sfirst[t][L]);
            dst[i] = e;
        }
    }
    __syncthreads();
    int off = 0;
    for (int u = 0; u < t; ++u) off += 21 + snsym[u];
    const int nsym = snsym[t];
    uint8_t *seg = op.dht + (int64_t)f * DHT_BYTES + off;
    for (int b = lane; b < 21 + nsym; b += 32) {
        uint8_t v;
        if (b < 4) v = b == 0 ? 0xFF : b == 1 ? 0xC4 : b == 2 ? (uint8_t)((19 + nsym) >> 8) : (uint8_t)(19 + nsym);
        else if (b == 4) v = (uint8_t)(((t & 1) << 4) | (t >> 1));
        else if (b < 21) v = (uint8_t)sbits[t][b - 4];
        else v = sval[t][b - 21];
        seg[b] = v;
    }
    if (threadIdx.x == 0) op.dhtlen[f] = 4 * 21 + snsym[0] + snsym[1] + snsym[2] + snsym[3];
}

// the zigzag nonzero mask of a block's AC coefficients
__device__ __forceinline__ uint64_t ac_mask(const int16_t *cf) {
    uint64_t mask = 0;
#pragma unroll
    for (int q = 0; q < 8; ++q) {
        const int4 v = __ldg(reinterpret_cast<const int4 *>(cf) + q);
        const int u[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            mask |= (uint64_t)((u[k] & 0xffff) != 0) << (q * 8 + 2 * k);
            mask |= (uint64_t)((u[k] >> 16) != 0) << (q * 8 + 2 * k + 1);
        }
    }
    return mask & ~1ull;
}

// Code length of every block from the frame's codes (OPT): what jpeg_transform writes in the standard mode
__global__ void __launch_bounds__(256) jpeg_blen_kernel(Geo g, Work w, Opt op) {
    __shared__ __align__(16) HuffTabs st;
    const int f = blockIdx.y;
    load_tabs(&st, op.tabs + f);
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= g.M * 6) return;
    const int64_t m = t / 6, fm = (int64_t)f * g.M + m;
    const int b = (int)(t - m * 6), tab = b >= 4;
    const int16_t *cf = w.coef + fm * 384 + b * 64;
    const Codes<true> c{st.dc, st.ac};
    uint64_t mask = ac_mask(cf);
    const int zrl = (int)(c.ac(tab, 0xF0) >> 16);
    int len = 0, prev = 0;
    while (mask) {
        const int zz = __ffsll((long long)mask) - 1;
        mask &= mask - 1;
        const int run = zz - prev - 1, s = nbits_of(__ldg(cf + zz));
        len += (run >> 4) * zrl + (int)(c.ac(tab, ((run & 15) << 4) | s) >> 16) + s;
        prev = zz;
    }
    if (prev != 63) len += (int)(c.ac(tab, 0) >> 16);
    if (b >= 1 && b <= 3) len += dc_len(c, 0, __ldg(cf) - __ldg(cf - 64));
    w.blen[fm * 8 + b] = (uint16_t)len;
}

template <bool OPT>
__global__ void __launch_bounds__(SCAN_THREADS) jpeg_mcu_scan_kernel(Geo g, Work w, Opt op) {
    const int f = blockIdx.x;
    const int64_t fm0 = (int64_t)f * g.M;
    Codes<OPT> c{};
    if constexpr (OPT) {
        __shared__ uint32_t sdc[2][16];
        if (threadIdx.x < 32) sdc[threadIdx.x >> 4][threadIdx.x & 15] = op.tabs[f].dc[threadIdx.x >> 4][threadIdx.x & 15];
        __syncthreads();
        c.dct = sdc;
    }
    const uint64_t total = block_scan(
        g.M,
        [&](int64_t m) -> uint64_t {
            const int4 l = *reinterpret_cast<const int4 *>(w.blen + (fm0 + m) * 8);
            const uint32_t u[4] = {(uint32_t)l.x, (uint32_t)l.y, (uint32_t)l.z, (uint32_t)l.w};
            uint32_t s = 0;
#pragma unroll
            for (int k = 0; k < 3; ++k) s += (u[k] & 0xffffu) + (u[k] >> 16);
            return s + cross_dc_len(c, load_dc(w.dcs + (fm0 + m) * 8), prev_dc(w.dcs, fm0 + m, m));
        },
        [&](int64_t m, uint64_t e) { w.off[fm0 + m] = e; });
    if (threadIdx.x == 0) w.bits[f] = total;
}

__global__ void jpeg_zero_kernel(Geo g, Work w, int n) {
    const int64_t gs = (int64_t)gridDim.x * blockDim.x;
    for (int f = 0; f < n; ++f) {
        const uint64_t tb = w.bits[f];
        const int64_t nw = (int64_t)((tb + 31) >> 5);
        const int pad = (int)(-(int64_t)tb & 7);
        uint32_t *wd = w.words + (int64_t)f * (g.wbytes / 4);
        for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nw; i += gs) {
            uint32_t v = 0;
            if (pad && i == (int64_t)(tb >> 5)) v = ((1u << pad) - 1u) << (32 - (int)(tb & 31) - pad);   // jchuff.c flush_bits
            wd[i] = v;
        }
    }
}

struct BitWriter {
    uint32_t *wd;
    int64_t widx;
    uint64_t acc;
    int nacc;
    __device__ BitWriter(uint32_t *words, uint64_t pos) : wd(words), widx((int64_t)(pos >> 5)), acc(0), nacc((int)(pos & 31)) {}
    __device__ __forceinline__ void put(uint32_t code, int len) {      // len <= 27
        acc = (acc << len) | code;
        nacc += len;
        if (nacc >= 32) {
            nacc -= 32;
            atomicOr(wd + widx++, (uint32_t)(acc >> nacc));
            acc &= (1ull << nacc) - 1ull;
        }
    }
    __device__ __forceinline__ void flush() {
        if (nacc > 0) atomicOr(wd + widx, (uint32_t)(acc << (32 - nacc)));
    }
};

__device__ __forceinline__ void put_value(BitWriter &bw, uint32_t hc, int v, int s) {
    const uint32_t extra = (uint32_t)(v < 0 ? v - 1 : v) & ((1u << s) - 1u);
    bw.put(((hc & 0xffffu) << s) | extra, (int)(hc >> 16) + s);
}

template <bool OPT>
__global__ void __launch_bounds__(256) jpeg_emit_kernel(Geo g, Work w, Opt op) {
    Codes<OPT> c{};
    if constexpr (OPT) {
        __shared__ __align__(16) HuffTabs st;
        load_tabs(&st, op.tabs + blockIdx.y);
        c = Codes<OPT>{st.dc, st.ac};
    }
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= g.M * 6) return;
    const int f = blockIdx.y;
    const int64_t m = t / 6, fm = (int64_t)f * g.M + m;
    const int b = (int)(t - m * 6);
    const Dc8 d = load_dc(w.dcs + fm * 8), p = prev_dc(w.dcs, fm, m);
    uint64_t pos = w.off[fm];
    int dcv = 0, pred = 0;
#pragma unroll
    for (int k = 0; k < 6; ++k) {                  // predictors: Y00 <- previous Y11, Y01..Y11 <- the block before, Cb / Cr <- previous
        const int pk = k == 0 ? p.v[3] : (k < 4 ? d.v[k - 1] : p.v[k]);
        if (k < b) {
            pos += w.blen[fm * 8 + k];
            if (k == 0 || k >= 4) pos += dc_len(c, k >= 4, d.v[k] - pk);
        }
        if (k == b) {
            dcv = d.v[k];
            pred = pk;
        }
    }
    const int16_t *cf = w.coef + fm * 384 + b * 64;
    uint64_t mask = ac_mask(cf);
    const int tab = b >= 4;
    BitWriter bw(w.words + (int64_t)f * (g.wbytes / 4), pos);
    const int diff = dcv - pred;
    put_value(bw, c.dc(tab, nbits_of(diff)), diff, nbits_of(diff));
    int prev = 0;
    while (mask) {
        const int zz = __ffsll((long long)mask) - 1;
        mask &= mask - 1;
        int run = zz - prev - 1;
        for (; run >= 16; run -= 16) bw.put(c.ac(tab, 0xF0) & 0xffffu, (int)(c.ac(tab, 0xF0) >> 16));
        const int v = __ldg(cf + zz), s = nbits_of(v);
        put_value(bw, c.ac(tab, (run << 4) | s), v, s);
        prev = zz;
    }
    if (prev != 63) bw.put(c.ac(tab, 0) & 0xffffu, (int)(c.ac(tab, 0) >> 16));
    bw.flush();
}

__device__ __forceinline__ int64_t entropy_bytes(uint64_t bits) { return (int64_t)((bits + 7) >> 3); }

__global__ void jpeg_ff_count_kernel(Geo g, Work w, int n) {
    const int64_t gs = (int64_t)gridDim.x * blockDim.x;
    for (int f = 0; f < n; ++f) {
        const int64_t nw = (int64_t)((w.bits[f] + 31) >> 5), nch = (nw + 3) >> 2;
        const uint4 *src = reinterpret_cast<const uint4 *>(w.words + (int64_t)f * (g.wbytes / 4));
        for (int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; c < nch; c += gs) {
            const uint4 v = src[c];
            const uint32_t u[4] = {v.x, v.y, v.z, v.w};
            uint32_t cnt = 0;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                if (c * 4 + k >= nw) break;          // words past the stream were never cleared
#pragma unroll
                for (int s = 0; s < 4; ++s) cnt += ((u[k] >> (8 * s)) & 0xffu) == 0xffu;
            }
            w.ffcnt[(int64_t)f * g.chunks + c] = cnt;
        }
    }
}

// OPT: hdr holds the header prefix (hlen bytes), then the SOS segment (op.slen bytes); the frame's DHT segments go between
template <bool OPT>
__global__ void __launch_bounds__(SCAN_THREADS) jpeg_ff_scan_kernel(Geo g, Work w, Header hdr, int hlen, uint8_t *out,
                                                                   int64_t slot, int64_t *lengths, Opt op) {
    const int f = blockIdx.x;
    const int64_t nbytes = entropy_bytes(w.bits[f]), nch = (nbytes + CHUNK - 1) / CHUNK;
    uint32_t *cnt = w.ffcnt + (int64_t)f * g.chunks;
    const uint64_t ff = block_scan(
        nch, [&](int64_t c) -> uint64_t { return cnt[c]; }, [&](int64_t c, uint64_t e) { cnt[c] = (uint32_t)e; });
    uint8_t *dst = out + (int64_t)f * slot;
    if constexpr (OPT) {
        const int dl = op.dhtlen[f], plen = hlen;
        const uint8_t *dht = op.dht + (int64_t)f * DHT_BYTES;
        hlen = plen + dl + op.slen;
        for (int i = threadIdx.x; i < hlen; i += blockDim.x)
            dst[i] = i < plen ? hdr.b[i] : i < plen + dl ? dht[i - plen] : hdr.b[i - dl];
        if (threadIdx.x == 0) op.hlen[f] = hlen;
    } else {
        for (int i = threadIdx.x; i < hlen; i += blockDim.x) dst[i] = hdr.b[i];
    }
    if (threadIdx.x == 0) {
        const int64_t end = hlen + nbytes + (int64_t)ff;
        dst[end] = 0xFF;
        dst[end + 1] = 0xD9;
        lengths[f] = end + 2;
    }
}

// OPT: each frame's data starts after its own header (op.hlen, from jpeg_ff_scan)
template <bool OPT>
__global__ void jpeg_stuff_kernel(Geo g, Work w, int n, int hlen, uint8_t *out, int64_t slot, Opt op) {
    const int64_t gs = (int64_t)gridDim.x * blockDim.x;
    for (int f = 0; f < n; ++f) {
        const int64_t nbytes = entropy_bytes(w.bits[f]), nch = (nbytes + CHUNK - 1) / CHUNK;
        const uint32_t *wd = w.words + (int64_t)f * (g.wbytes / 4);
        uint8_t *dst = out + (int64_t)f * slot + (OPT ? op.hlen[f] : hlen);
        for (int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; c < nch; c += gs) {
            int64_t o = c * CHUNK + w.ffcnt[(int64_t)f * g.chunks + c];
            const int nb = (int)min((int64_t)CHUNK, nbytes - c * CHUNK);
            for (int i = 0; i < nb; ++i) {
                const uint32_t word = wd[c * 4 + (i >> 2)];
                const uint8_t byte = (uint8_t)(word >> (24 - 8 * (i & 3)));
                dst[o++] = byte;
                if (byte == 0xFF) dst[o++] = 0;
            }
        }
    }
}

bool dims_ok(int H, int W) { return H >= 1 && H <= 65535 && W >= 1 && W <= 65535; }

// the optimized header (prefix, at most DHT_LEN_MAX bytes of DHT segments, SOS) fits AVB_JPEG_HEADER_MAX, which the slot
// bound counts
bool prefix_len_ok(int prefix_len, int sos_len) {
    return prefix_len >= 2 && sos_len >= 2 && prefix_len <= AVB_JPEG_HEADER_MAX &&
           sos_len <= AVB_JPEG_HEADER_MAX - DHT_LEN_MAX - prefix_len;
}

}  // namespace

extern "C" int64_t avb_jpeg_bound_bytes(int H, int W) {
    if (!dims_ok(H, W)) {
        avb::set_error("avb_jpeg_bound_bytes: H and W must lie in [1, 65535]");
        return AVB_E_ARG;
    }
    // header, every entropy byte stuffed (each may be 0xFF), EOI
    return AVB_JPEG_HEADER_MAX + 2 * geometry(H, W).wbytes + 2;
}

extern "C" int64_t avb_jpeg_workspace_bytes(int n, int H, int W) {
    if (!dims_ok(H, W) || n < 1 || n > 65535) {
        avb::set_error("avb_jpeg_workspace_bytes: bad geometry");
        return AVB_E_ARG;
    }
    return carve(geometry(H, W), n, nullptr, nullptr);
}

extern "C" int64_t avb_jpeg_opt_workspace_bytes(int n, int H, int W) {
    if (!dims_ok(H, W) || n < 1 || n > 65535) {
        avb::set_error("avb_jpeg_opt_workspace_bytes: bad geometry");
        return AVB_E_ARG;
    }
    return carve_opt(geometry(H, W), n, nullptr, nullptr);
}

namespace {

// AVB_REQUIRE with the name of the entry point that was called
#define K8_REQUIRE(cond, msg)                   \
    do {                                        \
        if (!(cond)) {                          \
            avb::set_error("%s: %s", fn, msg);  \
            return AVB_E_ARG;                   \
        }                                       \
    } while (0)

// OPT: header_host is the prefix before the DHT segments, sos_host the SOS segment
template <bool RGB, bool OPT>
int encode(const char *fn, const uint8_t *in, int n, int H, int W, int64_t in_frame_stride, int64_t in_row_stride,
           const uint8_t *header_host, int header_len, const uint8_t *sos_host, int sos_len, const uint8_t *qtables_host,
           uint8_t *out, int64_t out_slot_stride, int64_t *out_lengths_dev, void *workspace_dev, avb_stream_t stream) {
    K8_REQUIRE(in && header_host && (sos_host || !OPT) && qtables_host && out && out_lengths_dev && workspace_dev,
               "null pointer");
    K8_REQUIRE(n >= 1 && n <= 65535 && dims_ok(H, W), "n must lie in [1, 65535], H and W in [1, 65535]");
    K8_REQUIRE(in_row_stride >= 3LL * W && (n == 1 || in_frame_stride >= in_row_stride * (H - 1) + 3LL * W),
                "input strides overlap");
    if constexpr (OPT)
        K8_REQUIRE(prefix_len_ok(header_len, sos_len),
                   "prefix_len and sos_len must be at least 2, prefix_len + sos_len + 432 at most AVB_JPEG_HEADER_MAX");
    else
        K8_REQUIRE(header_len >= 2 && header_len <= AVB_JPEG_HEADER_MAX, "header_len must lie in [2, AVB_JPEG_HEADER_MAX]");
    K8_REQUIRE(out_slot_stride >= avb_jpeg_bound_bytes(H, W), "output slot smaller than avb_jpeg_bound_bytes(H, W)");
    K8_REQUIRE(((uintptr_t)workspace_dev & 15) == 0, "workspace must be 16-byte aligned");
    const Geo g = geometry(H, W);
    K8_REQUIRE(g.mh <= 65535, "too many MCU rows");
    QDiv qd;
    for (int t = 0; t < 2; ++t)
        for (int zz = 0; zz < 64; ++zz) {
            const int q = qtables_host[t * 64 + zz];
            K8_REQUIRE(q >= 1, "quantiser entries must lie in [1, 255]");
        }
    static const uint8_t zigzag[64] = {0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,  12, 19, 26, 33, 40, 48,
                                       41, 34, 27, 20, 13, 6,  7,  14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23,
                                       30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};
    for (int t = 0; t < 2; ++t)
        for (int zz = 0; zz < 64; ++zz) qd.d[t][zigzag[zz]] = (uint16_t)(8 * qtables_host[t * 64 + zz]);
    Header hdr;
    memcpy(hdr.b, header_host, header_len);
    Work w;
    carve(g, n, (uint8_t *)workspace_dev, &w);
    Opt op{};
    if constexpr (OPT) {
        memcpy(hdr.b + header_len, sos_host, sos_len);
        carve_opt(g, n, (uint8_t *)workspace_dev, &op);
        op.slen = sos_len;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const int grid = avb::sm_count() * 4;
    const unsigned block_ctas = (unsigned)((g.M * 6 + 255) / 256);
    if constexpr (OPT) AVB_CUDA_OK(cudaMemsetAsync(op.freq, 0, (size_t)n * 4 * 256 * 8, st));
    {
        AVB_TIMED("jpeg_transform", st);
        jpeg_transform_kernel<RGB, OPT><<<dim3((g.mw + STRIP - 1) / STRIP, g.mh, n), TF_THREADS, 0, st>>>(
            in, in_frame_stride, in_row_stride, g, qd, w, op);
    }
    if constexpr (OPT) {
        {
            AVB_TIMED("jpeg_dc_hist", st);
            jpeg_dc_hist_kernel<<<dim3((unsigned)((g.M + 255) / 256), n), 256, 0, st>>>(g, w, op);
        }
        {
            AVB_TIMED("jpeg_tables", st);
            jpeg_tables_kernel<<<n, 128, 0, st>>>(op);
        }
        {
            AVB_TIMED("jpeg_blen", st);
            jpeg_blen_kernel<<<dim3(block_ctas, n), 256, 0, st>>>(g, w, op);
        }
    }
    {
        AVB_TIMED("jpeg_mcu_scan", st);
        jpeg_mcu_scan_kernel<OPT><<<n, SCAN_THREADS, 0, st>>>(g, w, op);
    }
    {
        AVB_TIMED("jpeg_zero", st);
        jpeg_zero_kernel<<<grid, 256, 0, st>>>(g, w, n);
    }
    {
        AVB_TIMED("jpeg_emit", st);
        jpeg_emit_kernel<OPT><<<dim3(block_ctas, n), 256, 0, st>>>(g, w, op);
    }
    {
        AVB_TIMED("jpeg_ff_count", st);
        jpeg_ff_count_kernel<<<grid, 256, 0, st>>>(g, w, n);
    }
    {
        AVB_TIMED("jpeg_ff_scan", st);
        jpeg_ff_scan_kernel<OPT><<<n, SCAN_THREADS, 0, st>>>(g, w, hdr, header_len, out, out_slot_stride, out_lengths_dev,
                                                            op);
    }
    {
        AVB_TIMED("jpeg_stuff", st);
        jpeg_stuff_kernel<OPT><<<grid, 256, 0, st>>>(g, w, n, header_len, out, out_slot_stride, op);
    }
    AVB_CUDA_OK(cudaGetLastError());
    return AVB_OK;
}

#undef K8_REQUIRE

}  // namespace

extern "C" int avb_jpeg_encode_u8(const uint8_t *in, int n, int H, int W, int64_t in_frame_stride, int64_t in_row_stride,
                                  const uint8_t *header_host, int header_len, const uint8_t *qtables_host, uint8_t *out,
                                  int64_t out_slot_stride, int64_t *out_lengths_dev, void *workspace_dev,
                                  avb_stream_t stream) {
    return encode<false, false>(__func__, in, n, H, W, in_frame_stride, in_row_stride, header_host, header_len, nullptr, 0,
                                qtables_host, out, out_slot_stride, out_lengths_dev, workspace_dev, stream);
}

extern "C" int avb_jpeg_encode_rgb_u8(const uint8_t *in, int n, int H, int W, int64_t in_frame_stride,
                                      int64_t in_row_stride, const uint8_t *header_host, int header_len,
                                      const uint8_t *qtables_host, uint8_t *out, int64_t out_slot_stride,
                                      int64_t *out_lengths_dev, void *workspace_dev, avb_stream_t stream) {
    return encode<true, false>(__func__, in, n, H, W, in_frame_stride, in_row_stride, header_host, header_len, nullptr, 0,
                               qtables_host, out, out_slot_stride, out_lengths_dev, workspace_dev, stream);
}

extern "C" int avb_jpeg_opt_encode_u8(const uint8_t *in, int n, int H, int W, int64_t in_frame_stride,
                                      int64_t in_row_stride, const uint8_t *prefix_host, int prefix_len,
                                      const uint8_t *sos_host, int sos_len, const uint8_t *qtables_host, uint8_t *out,
                                      int64_t out_slot_stride, int64_t *out_lengths_dev, void *workspace_dev,
                                      avb_stream_t stream) {
    return encode<false, true>(__func__, in, n, H, W, in_frame_stride, in_row_stride, prefix_host, prefix_len, sos_host,
                               sos_len, qtables_host, out, out_slot_stride, out_lengths_dev, workspace_dev, stream);
}

extern "C" int avb_jpeg_opt_encode_rgb_u8(const uint8_t *in, int n, int H, int W, int64_t in_frame_stride,
                                          int64_t in_row_stride, const uint8_t *prefix_host, int prefix_len,
                                          const uint8_t *sos_host, int sos_len, const uint8_t *qtables_host, uint8_t *out,
                                          int64_t out_slot_stride, int64_t *out_lengths_dev, void *workspace_dev,
                                          avb_stream_t stream) {
    return encode<true, true>(__func__, in, n, H, W, in_frame_stride, in_row_stride, prefix_host, prefix_len, sos_host,
                              sos_len, qtables_host, out, out_slot_stride, out_lengths_dev, workspace_dev, stream);
}
