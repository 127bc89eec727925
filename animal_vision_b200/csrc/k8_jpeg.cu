// K8 -- batched baseline JPEG encoder, byte-identical to cv2.imencode(".jpg") with OpenCV's defaults
// (libjpeg-turbo: 4:2:0, standard Huffman tables, no restart interval).  Every stage is integer arithmetic, so
// the device restates libjpeg bit for bit (oracle/jpeg.py is the NumPy statement of the same stages):
//   jpeg_transform  one CTA per strip of 8 MCUs (16 x 128 px): BGR gather with edge replication, jccolor.c
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

__device__ __forceinline__ int nbits_of(int v) {
    v = abs(v);
    return v ? 32 - __clz(v) : 0;
}

__device__ __forceinline__ int dc_len(int tab, int diff) {
    const int s = nbits_of(diff);
    return (int)(c_huff.dc[tab][s] >> 16) + s;
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

__global__ void __launch_bounds__(TF_THREADS) jpeg_transform_kernel(const uint8_t *__restrict__ in, int64_t fs, int64_t rs,
                                                                     Geo g, QDiv qd, Work w) {
    __shared__ uint8_t sY[16][128], sCb[16][128], sCr[16][128], sC[2][8][64];
    __shared__ int work[STRIP * 6][8][9];
    __shared__ __align__(16) int16_t qz[STRIP * 6][64];
    __shared__ uint16_t sdiv[2][64];
    __shared__ uint8_t sizz[64];
    const int tid = threadIdx.x, f = blockIdx.z, my = blockIdx.y, mx0 = blockIdx.x * STRIP;
    if (tid < 128) sdiv[tid >> 6][tid & 63] = qd.d[tid >> 6][tid & 63];
    if (tid < 64) sizz[tid] = c_izz[tid];
    const uint8_t *fin = in + (int64_t)f * fs;
    for (int p = tid; p < 16 * 128; p += TF_THREADS) {          // columns / rows past the edge repeat the last one
        const int r = p >> 7, c = p & 127;
        const int gy = min(my * 16 + r, g.H - 1), gx = min(mx0 * 16 + c, g.W - 1);
        const uint8_t *px = fin + gy * rs + gx * 3;
        const int b = px[0], gg = px[1], rr = px[2];              // BGR
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
        if (b >= 1 && b <= 3) len += dc_len(0, qz[bl][0] - qz[bl - 1][0]);
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
__device__ __forceinline__ int cross_dc_len(const Dc8 &d, const Dc8 &p) {
    return dc_len(0, d.v[0] - p.v[3]) + dc_len(1, d.v[4] - p.v[4]) + dc_len(1, d.v[5] - p.v[5]);
}

__device__ __forceinline__ Dc8 prev_dc(const int16_t *dcs, int64_t fm, int64_t m) {
    if (m > 0) return load_dc(dcs + (fm - 1) * 8);
    Dc8 z;
#pragma unroll
    for (int k = 0; k < 8; ++k) z.v[k] = 0;
    return z;
}

__global__ void __launch_bounds__(SCAN_THREADS) jpeg_mcu_scan_kernel(Geo g, Work w) {
    const int f = blockIdx.x;
    const int64_t fm0 = (int64_t)f * g.M;
    const uint64_t total = block_scan(
        g.M,
        [&](int64_t m) -> uint64_t {
            const int4 l = *reinterpret_cast<const int4 *>(w.blen + (fm0 + m) * 8);
            const uint32_t u[4] = {(uint32_t)l.x, (uint32_t)l.y, (uint32_t)l.z, (uint32_t)l.w};
            uint32_t s = 0;
#pragma unroll
            for (int k = 0; k < 3; ++k) s += (u[k] & 0xffffu) + (u[k] >> 16);
            return s + cross_dc_len(load_dc(w.dcs + (fm0 + m) * 8), prev_dc(w.dcs, fm0 + m, m));
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

__global__ void __launch_bounds__(256) jpeg_emit_kernel(Geo g, Work w) {
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
            if (k == 0 || k >= 4) pos += dc_len(k >= 4, d.v[k] - pk);
        }
        if (k == b) {
            dcv = d.v[k];
            pred = pk;
        }
    }
    const int16_t *cf = w.coef + fm * 384 + b * 64;
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
    mask &= ~1ull;
    const int tab = b >= 4;
    BitWriter bw(w.words + (int64_t)f * (g.wbytes / 4), pos);
    const int diff = dcv - pred;
    put_value(bw, c_huff.dc[tab][nbits_of(diff)], diff, nbits_of(diff));
    int prev = 0;
    while (mask) {
        const int zz = __ffsll((long long)mask) - 1;
        mask &= mask - 1;
        int run = zz - prev - 1;
        for (; run >= 16; run -= 16) bw.put(c_huff.ac[tab][0xF0] & 0xffffu, (int)(c_huff.ac[tab][0xF0] >> 16));
        const int v = __ldg(cf + zz), s = nbits_of(v);
        put_value(bw, c_huff.ac[tab][(run << 4) | s], v, s);
        prev = zz;
    }
    if (prev != 63) bw.put(c_huff.ac[tab][0] & 0xffffu, (int)(c_huff.ac[tab][0] >> 16));
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

__global__ void __launch_bounds__(SCAN_THREADS) jpeg_ff_scan_kernel(Geo g, Work w, Header hdr, int hlen, uint8_t *out,
                                                                   int64_t slot, int64_t *lengths) {
    const int f = blockIdx.x;
    const int64_t nbytes = entropy_bytes(w.bits[f]), nch = (nbytes + CHUNK - 1) / CHUNK;
    uint32_t *cnt = w.ffcnt + (int64_t)f * g.chunks;
    const uint64_t ff = block_scan(
        nch, [&](int64_t c) -> uint64_t { return cnt[c]; }, [&](int64_t c, uint64_t e) { cnt[c] = (uint32_t)e; });
    uint8_t *dst = out + (int64_t)f * slot;
    for (int i = threadIdx.x; i < hlen; i += blockDim.x) dst[i] = hdr.b[i];
    if (threadIdx.x == 0) {
        const int64_t end = hlen + nbytes + (int64_t)ff;
        dst[end] = 0xFF;
        dst[end + 1] = 0xD9;
        lengths[f] = end + 2;
    }
}

__global__ void jpeg_stuff_kernel(Geo g, Work w, int n, int hlen, uint8_t *out, int64_t slot) {
    const int64_t gs = (int64_t)gridDim.x * blockDim.x;
    for (int f = 0; f < n; ++f) {
        const int64_t nbytes = entropy_bytes(w.bits[f]), nch = (nbytes + CHUNK - 1) / CHUNK;
        const uint32_t *wd = w.words + (int64_t)f * (g.wbytes / 4);
        uint8_t *dst = out + (int64_t)f * slot + hlen;
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

extern "C" int avb_jpeg_encode_u8(const uint8_t *in, int n, int H, int W, int64_t in_frame_stride, int64_t in_row_stride,
                                  const uint8_t *header_host, int header_len, const uint8_t *qtables_host, uint8_t *out,
                                  int64_t out_slot_stride, int64_t *out_lengths_dev, void *workspace_dev,
                                  avb_stream_t stream) {
    AVB_REQUIRE(in && header_host && qtables_host && out && out_lengths_dev && workspace_dev, "null pointer");
    AVB_REQUIRE(n >= 1 && n <= 65535 && dims_ok(H, W), "n must lie in [1, 65535], H and W in [1, 65535]");
    AVB_REQUIRE(in_row_stride >= 3LL * W && (n == 1 || in_frame_stride >= in_row_stride * (H - 1) + 3LL * W),
                "input strides overlap");
    AVB_REQUIRE(header_len >= 2 && header_len <= AVB_JPEG_HEADER_MAX, "header_len must lie in [2, AVB_JPEG_HEADER_MAX]");
    AVB_REQUIRE(out_slot_stride >= avb_jpeg_bound_bytes(H, W), "output slot smaller than avb_jpeg_bound_bytes(H, W)");
    AVB_REQUIRE(((uintptr_t)workspace_dev & 15) == 0, "workspace must be 16-byte aligned");
    const Geo g = geometry(H, W);
    AVB_REQUIRE(g.mh <= 65535, "too many MCU rows");
    QDiv qd;
    for (int t = 0; t < 2; ++t)
        for (int zz = 0; zz < 64; ++zz) {
            const int q = qtables_host[t * 64 + zz];
            AVB_REQUIRE(q >= 1, "quantiser entries must lie in [1, 255]");
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
    cudaStream_t st = (cudaStream_t)stream;
    const int grid = avb::sm_count() * 4;
    {
        AVB_TIMED("jpeg_transform", st);
        jpeg_transform_kernel<<<dim3((g.mw + STRIP - 1) / STRIP, g.mh, n), TF_THREADS, 0, st>>>(in, in_frame_stride,
                                                                                              in_row_stride, g, qd, w);
    }
    {
        AVB_TIMED("jpeg_mcu_scan", st);
        jpeg_mcu_scan_kernel<<<n, SCAN_THREADS, 0, st>>>(g, w);
    }
    {
        AVB_TIMED("jpeg_zero", st);
        jpeg_zero_kernel<<<grid, 256, 0, st>>>(g, w, n);
    }
    {
        AVB_TIMED("jpeg_emit", st);
        jpeg_emit_kernel<<<dim3((unsigned)((g.M * 6 + 255) / 256), n), 256, 0, st>>>(g, w);
    }
    {
        AVB_TIMED("jpeg_ff_count", st);
        jpeg_ff_count_kernel<<<grid, 256, 0, st>>>(g, w, n);
    }
    {
        AVB_TIMED("jpeg_ff_scan", st);
        jpeg_ff_scan_kernel<<<n, SCAN_THREADS, 0, st>>>(g, w, hdr, header_len, out, out_slot_stride, out_lengths_dev);
    }
    {
        AVB_TIMED("jpeg_stuff", st);
        jpeg_stuff_kernel<<<grid, 256, 0, st>>>(g, w, n, header_len, out, out_slot_stride);
    }
    AVB_CUDA_OK(cudaGetLastError());
    return AVB_OK;
}
