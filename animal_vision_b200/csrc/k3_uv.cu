// K3: the UV path -- RGB -> analytic 31-band spectrum -> photoreceptor catches -> von Kries
// adaptation -> small acuity blur -> (U,B,G) visualisation map with GLOBAL percentiles -> sRGB
// encode, without ever materialising the H x W x 31 hyperspectral cube (257 MB per 1080p frame in
// the reference: classic_rgb_to_hsi.py:47-82, honeybee.py:126-135).
//
// The global statistics force several passes over the frame; every pass RE-COMPUTES the receptor
// catches from the uint8 input (3 B/px from HBM per pass: a 20-frame launch is 498 MB, far beyond the 126 MB L2; running
// frames in L2-sized groups was measured and is SLOWER -- 2.61 -> 3.06 / 3.72 / 5.73 ms per 20 4K frames for groups of
// 4 / 2 / 1, the passes are issue bound, not DRAM bound) instead of round-tripping fp32 planes through HBM:
//   stats    raw catches -> per-frame max and sum of each receptor          (white patch / gray world)
//   prep     (1 thread per frame) fold the adaptation into the receptor matrix, size the bins
//   hist     adapted + blurred catches -> mapper quantities -> 2048 linear bins per quantity
//            (+ the quantities themselves, 4 B per pixel, for the compact pass)
//   scan     locate the bin(s) that hold the two order statistics of every percentile request
//   compact  read back the quantity planes the hist pass wrote, append the values that fall into
//            those bins to a candidate list
//   select   exact radix select among the candidates -> numpy.percentile(method="linear")
//   map      recompute, apply the mapper, clip -> OETF -> uint8
// The percentile is EXACT (same order statistics numpy picks), whatever the value distribution:
// binning only decides how many candidates the select step sees.
//
// Pixel walk: one warp owns a strip of 120 output columns (lane l holds pixels 4l-4 .. 4l-1 of the
// strip, three aligned 32-bit loads per row) and streams down 64 rows; horizontal blur neighbours
// come from the adjacent lanes by shuffle, the vertical window lives in registers, so there is no
// shared-memory tile, no __syncthreads and no per-pixel index arithmetic.
//
// Receptor catches come either from the per-pixel band sum in registers ("bands" mode, the
// reference's own order of operations) or from the algebraically identical 3x3 (the whole chain
// lobes -> illuminant -> sensitivities is linear; SURVEY.md 8a-11: 1.9e-7 relative difference).
#include <algorithm>

#include "avb_common.cuh"

namespace avb {

constexpr int UV_BINS = 2048;
constexpr int UV_NH = 3;                 // histograms (mapper quantities) per frame
constexpr int UV_NR = 4;                 // percentile requests per frame
constexpr int UV_MAX_BANDS = 160;
constexpr int UV_THREADS = 256, UV_WARPS = UV_THREADS / 32;
#ifndef UV_RH_ROWS
#define UV_RH_ROWS 64
#endif
constexpr int UV_RH = UV_RH_ROWS;        // output rows per strip
#ifndef UV_MINB
#define UV_MINB 4
#endif
#ifndef UV_HIST_WAVES
#define UV_HIST_WAVES 1
#endif
constexpr unsigned FULL = 0xffffffffu;

enum { MAP_OPPONENT = 0, MAP_FALSECOLOR = 1, MAP_MATRIX = 2, MAP_PURPLE = 3, MAP_MIXED = 4 };
enum { QS_OPP = 0, QS_UBG = 1, QS_U = 2 };   // which quantities feed the histograms

struct UvFrameStats {
    uint32_t max_bits[3];
    uint32_t pad0;
    double sum[3];
    float rcp[3];                // correctly rounded reciprocals of the adaptation divisors
    float pad2[6];
    float scale[3];              // adaptation divisors
    float inv_w[UV_NH];          // bins per unit value
    uint32_t bin_lo[UV_NR], bin_hi[UV_NR], rank_lo[UV_NR], rank_hi[UV_NR], cand_count[UV_NR];
    float pct[UV_NR];
    uint32_t pad1;
};
static_assert(sizeof(UvFrameStats) % 8 == 0, "stats block must stay 8-byte aligned");

struct UvParams {
    FrameIO io;
    const float *lut;            // decode LUT (device, 256)
    float M3[9];                 // collapsed receptor matrix: catch k = sum_c M3[3k+c] * lin[c]
    const float *bands;          // bands mode: [B][8] = g0,g1,g2 (lobe of input channel c), E, s0,s1,s2, 0
    int n_bands;                 // 0 -> collapsed mode
    float denom_eps;             // lobe normaliser + 1e-8 (float32, as torch computes it)
    int adapt;                   // 0 none, 1 white patch (max), 2 gray world (mean)
    float eps;                   // 1e-8
    float t0, t1, t2;            // blur taps: centre, +-1, +-2
    UvFrameStats *stats;         // [n]
    uint32_t *hist;              // [n][UV_NH][UV_BINS]
    float *planes;               // [n][UV_NH][H*W]: mapper quantities written by the hist pass
    float *cand;                 // [n][n_req][cap]
    long long cap;
    const uint32_t *enc;
    int n_req;
    int req_hist[UV_NR];
    long long k_lo[UV_NR], k_hi[UV_NR];
    float gamma[UV_NR];
    int mapper;
    float map_m[9];              // MAP_MATRIX
    float anchors[6];            // MAP_PURPLE / MAP_MIXED: linear-light purple and warm anchors
    float mix_alpha;             // MAP_MIXED
    float *dbg_catches;          // optional [n][H][W][3] raw catches (test hook), else nullptr
    int aligned_in, aligned_out; // rows / frames 4-byte aligned -> 32-bit pixel-group accesses
    int strips_x, strips_y;
};

// x / s with r = RN(1/s): one Newton correction on the quotient (Markstein) gives the correctly
// rounded IEEE quotient for the value ranges here (no overflow / underflow), in 3 instructions.
// Exactness matters: a flat frame must adapt to exactly 1.0 in every receptor, as it does in the
// reference, or the opponent radius stops being exactly 0.
__device__ __forceinline__ float div_by(float x, float s, float r) {
    const float q = __fmul_rn(x, r);
    return fmaf(fmaf(-q, s, x), r, q);
}

// "bands" mode: classic_rgb_to_hsi.py:70-78, honeybee.py:126-135 in the reference's own order:
// spec = (g2*c2 + g1*c1 + g0*c0) / (denom+1e-8);  rad = spec * E;  catch += rad * s.
// Kept out of line: it is the fidelity mode, and inlining it four times per pixel group bloats
// every walker past the instruction cache.
__device__ __noinline__ void band_sum(const float4 *bands, int n_bands, float denom_eps, float c0, float c1, float c2,
                                      float &u, float &b, float &g) {
    float au = 0.f, ab = 0.f, ag = 0.f;
    for (int l = 0; l < n_bands; ++l) {
        const float4 lo = __ldg(bands + 2 * l), hi = __ldg(bands + 2 * l + 1);
        float spec = __fadd_rn(__fadd_rn(__fmul_rn(lo.z, c2), __fmul_rn(lo.y, c1)), __fmul_rn(lo.x, c0));
        spec = fmaxf(__fdiv_rn(spec, denom_eps), 0.f);
        const float rad = __fmul_rn(spec, lo.w);
        au = fmaf(rad, hi.x, au);
        ab = fmaf(rad, hi.y, ab);
        ag = fmaf(rad, hi.z, ag);
    }
    u = au; b = ab; g = ag;
}

// ------------------------------------------------------------------ per-pixel receptor catches
template <bool BANDS>
struct Catcher {
    const float *lut_s;
    float m[9];
    const float4 *bands;
    int n_bands;
    float denom_eps;
    float sc[3], rc[3];
    bool divide;

    __device__ __forceinline__ void init_raw(const UvParams &p, const float *lut) {
        lut_s = lut;
#pragma unroll
        for (int i = 0; i < 9; ++i) m[i] = p.M3[i];
        bands = reinterpret_cast<const float4 *>(p.bands);
        n_bands = p.n_bands;
        denom_eps = p.denom_eps;
        sc[0] = sc[1] = sc[2] = 1.f;
        rc[0] = rc[1] = rc[2] = 1.f;
        divide = false;
    }
    __device__ __forceinline__ void init_adapted(const UvParams &p, const UvFrameStats &st, const float *lut) {
        init_raw(p, lut);
#pragma unroll
        for (int k = 0; k < 3; ++k) { sc[k] = st.scale[k]; rc[k] = st.rcp[k]; }
        divide = p.adapt != 0;
    }
    __device__ __forceinline__ void operator()(uint32_t b0, uint32_t b1, uint32_t b2, float &u, float &b, float &g) const {
        from_linear(lut_s[b0], lut_s[b1], lut_s[b2], u, b, g);
    }
    // catches of one pixel from its linear-light channels (the float-frame path decodes with powf instead of the LUT)
    __device__ __forceinline__ void from_linear(float c0, float c1, float c2, float &u, float &b, float &g) const {
        if constexpr (!BANDS) {
            u = m[0] * c0 + m[1] * c1 + m[2] * c2;
            b = m[3] * c0 + m[4] * c1 + m[5] * c2;
            g = m[6] * c0 + m[7] * c1 + m[8] * c2;
            if (divide) {      // uv_helpers.py:195-206: x / scale, correctly rounded (see div_by)
                u = div_by(u, sc[0], rc[0]);
                b = div_by(b, sc[1], rc[1]);
                g = div_by(g, sc[2], rc[2]);
            }
        } else {
            float au, ab, ag;
            band_sum(bands, n_bands, denom_eps, c0, c1, c2, au, ab, ag);
            if (divide) {      // uv_helpers.py:195-206: divide by the global max / mean
                au = __fdiv_rn(au, sc[0]);
                ab = __fdiv_rn(ab, sc[1]);
                ag = __fdiv_rn(ag, sc[2]);
            }
            u = au; b = ab; g = ag;
        }
    }
};

__device__ __forceinline__ uint32_t byte_k(uint32_t w, int k) { return __byte_perm(w, 0, 0x4440 + k); }

// 4 packed pixels (three 32-bit words) -> catches
template <class Cat>
__device__ __forceinline__ void catches4(const Cat &cat, const uint32_t (&w)[3], float (&c)[4][3]) {
    cat(byte_k(w[0], 0), byte_k(w[0], 1), byte_k(w[0], 2), c[0][0], c[0][1], c[0][2]);
    cat(byte_k(w[0], 3), byte_k(w[1], 0), byte_k(w[1], 1), c[1][0], c[1][1], c[1][2]);
    cat(byte_k(w[1], 2), byte_k(w[1], 3), byte_k(w[2], 0), c[2][0], c[2][1], c[2][2]);
    cat(byte_k(w[2], 1), byte_k(w[2], 2), byte_k(w[2], 3), c[3][0], c[3][1], c[3][2]);
}

// ------------------------------------------------------------------ the strip walk
// Calls op(y, gx, v, ok) once per output row for every lane: v[j][k] = adapted + blurred catch k of
// pixel (y, gx + j); ok is false for the two halo lanes.  All 32 lanes call op together.
template <int R, class Cat, class Op>
__device__ __forceinline__ void uv_walk(const UvParams &p, const Cat &cat, const uint8_t *src, int xs, int ys, int rows, Op &op) {
    constexpr int OFF = R ? 4 : 0;
    const int lane = threadIdx.x & 31;
    const int H = p.io.H, W = p.io.W;
    const int gx = xs - OFF + 4 * lane;
    const bool fast = p.aligned_in && gx >= 0 && gx + 3 < W;
    int xi[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) xi[j] = 3 * reflect101(gx + j, W);
    const bool lane_ok = (R == 0) || (lane >= 1 && lane <= 30);

    auto load = [&](int i, uint32_t(&w)[3]) {
        const uint8_t *row = src + (int64_t)reflect101(ys + i, H) * p.io.in_rs;
        if (fast) {
            const uint32_t *q = reinterpret_cast<const uint32_t *>(row + 3 * gx);
            w[0] = __ldg(q); w[1] = __ldg(q + 1); w[2] = __ldg(q + 2);
        } else {
            uint32_t b[12];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const uint8_t *q = row + xi[j];
                b[3 * j] = q[0]; b[3 * j + 1] = q[1]; b[3 * j + 2] = q[2];
            }
#pragma unroll
            for (int k = 0; k < 3; ++k) w[k] = b[4 * k] | (b[4 * k + 1] << 8) | (b[4 * k + 2] << 16) | (b[4 * k + 3] << 24);
        }
    };

    // Vertical pass in accumulator ("scatter") form: acc[m] is the partial sum of the output row
    // that still misses 2R - m input rows.  No rotating window, no per-phase unrolling, so the
    // per-pixel operator is instantiated once (the unrolled form thrashed the instruction cache).
    float acc[2 * R + 1][4][3];
#pragma unroll
    for (int m = 0; m < 2 * R + 1; ++m)
#pragma unroll
        for (int j = 0; j < 4; ++j)
#pragma unroll
            for (int k = 0; k < 3; ++k) acc[m][j][k] = 0.f;
    uint32_t w[3], wn[3] = {0u, 0u, 0u};
    const int n_iter = rows + 2 * R;
    const float tp[3] = {p.t0, p.t1, p.t2};
    load(-R, w);
    for (int i = 0; i < n_iter; ++i) {              // iteration i reads input row ys + i - R
        if (i + 1 < n_iter) load(i + 1 - R, wn);
        float c[4][3];
        catches4(cat, w, c);
        float v[4][3];
        if constexpr (R == 0) {
#pragma unroll
            for (int j = 0; j < 4; ++j)
#pragma unroll
                for (int k = 0; k < 3; ++k) v[j][k] = c[j][k];
        } else {
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                // horizontal pass (rows first, as cv2.GaussianBlur): neighbours from adjacent lanes
                float e[8];
                e[1] = __shfl_up_sync(FULL, c[3][k], 1);
                e[6] = __shfl_down_sync(FULL, c[0][k], 1);
                if (R == 2) {
                    e[0] = __shfl_up_sync(FULL, c[2][k], 1);
                    e[7] = __shfl_down_sync(FULL, c[1][k], 1);
                } else {
                    e[0] = e[7] = 0.f;
                }
#pragma unroll
                for (int j = 0; j < 4; ++j) e[2 + j] = c[j][k];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    float h = fmaf(tp[1], e[1 + j] + e[3 + j], tp[0] * e[2 + j]);
                    if (R == 2) h = fmaf(tp[2], e[j] + e[4 + j], h);
                    // vertical pass: finish the oldest output row, advance the others
                    v[j][k] = fmaf(tp[R], h, acc[0][j][k]);
#pragma unroll
                    for (int m = 0; m < 2 * R - 1; ++m) {
                        const int d = (R - 1 - m) < 0 ? -(R - 1 - m) : (R - 1 - m);
                        acc[m][j][k] = fmaf(tp[d], h, acc[m + 1][j][k]);
                    }
                    acc[2 * R - 1][j][k] = tp[R] * h;
                }
            }
        }
        if (i >= 2 * R) op(ys + i - 2 * R, gx, v, lane_ok);
#pragma unroll
        for (int k = 0; k < 3; ++k) w[k] = wn[k];
    }
}

// strip task -> (xs, ys, rows)
template <int R>
__device__ __forceinline__ void strip_of(const UvParams &p, int task, int &xs, int &ys, int &rows) {
    constexpr int SW = R ? 120 : 128;
    const int sy = task / p.strips_x, sx = task - sy * p.strips_x;
    xs = sx * SW;
    ys = sy * UV_RH;
    rows = min(UV_RH, p.io.H - ys);
}

// sqrt on the SFU (rsq + multiply, ~1 ulp): the opponent radius only feeds a percentile that is
// computed from the very same values and a saturation ratio, both insensitive at the 1e-7 level.
__device__ __forceinline__ float sqrt_sfu(float x) {
    float r;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}

// atan2 without branches: octant reduction + the degree-17 odd minimax polynomial of Abramowitz &
// Stegun 4.4.49 (|error| <= 2e-8 in exact arithmetic, 1.1e-7 evaluated in float32).  The hue only
// needs ~1e-6: an error e in the angle moves the output colour by <= e in linear light, i.e.
// < 1e-3 LSB after the encode.
__device__ __forceinline__ float atan2_fast(float y, float x) {
    const float ax = fabsf(x), ay = fabsf(y);
    const float mx = fmaxf(ax, ay), mn = fminf(ax, ay);
    const float a = mx > 0.f ? __fdividef(mn, mx) : 0.f;
    const float s = a * a;
    float r = 0.0028662257f;
    r = fmaf(r, s, -0.0161657367f);
    r = fmaf(r, s, 0.0429096138f);
    r = fmaf(r, s, -0.0752896400f);
    r = fmaf(r, s, 0.1065626393f);
    r = fmaf(r, s, -0.1420889944f);
    r = fmaf(r, s, 0.1999355085f);
    r = fmaf(r, s, -0.3333314528f);
    r = fmaf(r * s, a, a);
    r = ay > ax ? 1.57079632679489662f - r : r;
    r = x < 0.f ? 3.14159265358979324f - r : r;
    return y < 0.f ? -r : r;
}

// hue of the opponent mapper (uv_mappers.py:57-60): (atan2(O2, O1) + pi) / 2 pi, float32 constants as NumPy rounds them
template <bool PRECISE>
__device__ __forceinline__ float opp_hue(const float (&c)[3]) {
    const float O1 = c[2] - c[1], O2 = c[1] - c[0];
    const float PI_F = 3.14159274101257324f;          // float32(np.pi)
    const float ang = PRECISE ? atan2f(O2, O1) : atan2_fast(O2, O1);
    return div_by(__fadd_rn(ang, PI_F), 6.28318548202514648f, 0.159154936671257019f);
}

// ------------------------------------------------------------------ mapper quantities
// PRECISE (the float32 plane route, whose float outputs are compared at 1e-5): IEEE sqrt / libm atan2 instead of
// the SFU forms that are ample for uint8 outputs.
template <int QS, bool PRECISE = false>
__device__ __forceinline__ void quantities(const float (&c)[3], float (&q)[UV_NH]) {
    if (QS == QS_OPP) {
        // uv_mappers.py:55-60
        const float O1 = c[2] - c[1], O2 = c[1] - c[0];
        const float r2 = __fadd_rn(__fmul_rn(O1, O1), __fmul_rn(O2, O2));
        q[0] = PRECISE ? __fsqrt_rn(r2) : sqrt_sfu(r2);
        q[1] = div_by(__fadd_rn(__fadd_rn(c[0], c[1]), c[2]), 3.0f, 0.333333343267440796f);
        q[2] = 0.f;
    } else {
        q[0] = c[0]; q[1] = c[1]; q[2] = c[2];
    }
}
template <int QS>
struct QCount { static constexpr int value = QS == QS_OPP ? 2 : (QS == QS_UBG ? 3 : 1); };

__device__ __forceinline__ int bin_of(float v, float inv_w) {
    return min(UV_BINS - 1, max(0, __float2int_rd(v * inv_w)));
}

// ------------------------------------------------------------------ stats: maxima / sums of raw catches
template <bool BANDS>
// (no occupancy target: measured 0.265 ms as compiled, 0.284 / 0.321 / 0.355 / 0.393 ms with 4 / 5 / 6 / 8 CTAs per SM requested)
__global__ void __launch_bounds__(256) uv_stats_kernel(const __grid_constant__ UvParams p) {
    __shared__ float lut_s[256];
    for (int i = threadIdx.x; i < 256; i += blockDim.x) lut_s[i] = __ldg(p.lut + i);
    __syncthreads();
    const int frame = blockIdx.y;
    const uint8_t *src = p.io.in + (int64_t)frame * p.io.in_fs;
    Catcher<BANDS> cat;
    cat.init_raw(p, lut_s);
    float mx[3] = {0.f, 0.f, 0.f};
    double sm[3] = {0.0, 0.0, 0.0};
    const int W = p.io.W, H = p.io.H;
    const int groups = (W + 3) >> 2;
    for (int y = blockIdx.x; y < H; y += gridDim.x) {
        const uint8_t *row = src + (int64_t)y * p.io.in_rs;
        float rs[3] = {0.f, 0.f, 0.f};
        int gi = threadIdx.x;
        if (p.aligned_in) {
            // four independent pixel groups per thread in flight (the pass is latency bound otherwise)
            for (; gi + 3 * (int)blockDim.x < groups - 1; gi += 4 * blockDim.x) {
                uint32_t w[4][3];
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const uint32_t *q = reinterpret_cast<const uint32_t *>(row + 12 * (gi + u * (int)blockDim.x));
                    w[u][0] = __ldg(q); w[u][1] = __ldg(q + 1); w[u][2] = __ldg(q + 2);
                }
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    float c[4][3];
                    catches4(cat, w[u], c);
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
#pragma unroll
                        for (int k = 0; k < 3; ++k) {
                            mx[k] = fmaxf(mx[k], c[j][k]);
                            rs[k] += c[j][k];
                        }
                        if (p.dbg_catches) {
                            float *d = p.dbg_catches + (((int64_t)frame * H + y) * W + 4 * (gi + u * (int)blockDim.x) + j) * 3;
                            d[0] = c[j][0]; d[1] = c[j][1]; d[2] = c[j][2];
                        }
                    }
                }
            }
        }
        for (; gi < groups; gi += blockDim.x) {
            const int gx = 4 * gi;
            float c[4][3];
            int npx = min(4, W - gx);
            if (p.aligned_in && npx == 4) {
                const uint32_t *q = reinterpret_cast<const uint32_t *>(row + 3 * gx);
                const uint32_t w[3] = {__ldg(q), __ldg(q + 1), __ldg(q + 2)};
                catches4(cat, w, c);
            } else {
                for (int j = 0; j < npx; ++j) cat(row[3 * (gx + j)], row[3 * (gx + j) + 1], row[3 * (gx + j) + 2], c[j][0], c[j][1], c[j][2]);
            }
            for (int j = 0; j < npx; ++j) {
#pragma unroll
                for (int k = 0; k < 3; ++k) {
                    mx[k] = fmaxf(mx[k], c[j][k]);
                    rs[k] += c[j][k];
                }
                if (p.dbg_catches) {
                    float *d = p.dbg_catches + (((int64_t)frame * H + y) * W + gx + j) * 3;
                    d[0] = c[j][0]; d[1] = c[j][1]; d[2] = c[j][2];
                }
            }
        }
#pragma unroll
        for (int k = 0; k < 3; ++k) sm[k] += (double)rs[k];     // float partial per (thread,row): <= ~W/1024 terms
    }
    // block reduction first: one atomic per block and receptor, not one per warp
    __shared__ float red_m[8][3];
    __shared__ double red_s[8][3];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        float m = mx[k];
        double s = sm[k];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            m = fmaxf(m, __shfl_xor_sync(FULL, m, o));
            s += __shfl_xor_sync(FULL, s, o);
        }
        if (lane == 0) { red_m[wid][k] = m; red_s[wid][k] = s; }
    }
    __syncthreads();
    if (threadIdx.x < 3) {
        const int k = threadIdx.x;
        float m = 0.f;
        double s = 0.0;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) { m = fmaxf(m, red_m[w][k]); s += red_s[w][k]; }
        UvFrameStats &st = p.stats[frame];
        atomicMax(&st.max_bits[k], __float_as_uint(fmaxf(m, 0.f)));
        atomicAdd(&st.sum[k], s);
    }
}

// ------------------------------------------------------------------ prep: adaptation + bin widths
template <int QS>
__global__ void uv_prep_kernel(const __grid_constant__ UvParams p) {
    const int frame = blockIdx.x * blockDim.x + threadIdx.x;
    if (frame >= p.io.n) return;
    UvFrameStats &st = p.stats[frame];
    const double npx = (double)p.io.H * (double)p.io.W;
    float ub[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const float mx = __uint_as_float(st.max_bits[k]);
        float s = 1.0f;
        if (p.adapt == 1) s = fmaxf(mx, p.eps);                                  // uv_helpers.py:195-199
        else if (p.adapt == 2) s = fmaxf((float)(st.sum[k] / npx), p.eps);       // uv_helpers.py:202-206
        st.scale[k] = s;
        st.rcp[k] = __frcp_rn(s);
        ub[k] = mx / s * 1.001f + 1e-30f;
    }
    float hb[UV_NH];
    if (QS == QS_OPP) {
        const float a = fmaxf(ub[2], ub[1]), b = fmaxf(ub[1], ub[0]);
        hb[0] = sqrtf(a * a + b * b) * 1.001f;
        hb[1] = (ub[0] + ub[1] + ub[2]) * (1.001f / 3.0f);
        hb[2] = 1.f;
    } else {
        hb[0] = ub[0]; hb[1] = ub[1]; hb[2] = ub[2];
    }
#pragma unroll
    for (int h = 0; h < UV_NH; ++h) st.inv_w[h] = (float)UV_BINS / fmaxf(hb[h], 1e-30f);
}

// The map pass of every mapper with percentiles reads the planes of the hist pass -- (radius, L, hue) for the opponent mapper,
// the adapted, blurred catches themselves for the others -- when a lane's four pixels are one aligned float4 per plane and
// one aligned 12-byte group of the output (any other geometry, and the matrix mapper, take the second walk, uv_map_kernel).
__host__ __device__ __forceinline__ bool map_from_planes(const UvParams &p) {
    return p.n_req > 0 && (p.io.W & 3) == 0 && p.aligned_out != 0;
}

// ------------------------------------------------------------------ hist
template <int QS>
struct HistOp {
    uint32_t *hs;
    float *planes;               // this frame's [NQ][H*W] quantity planes (read back by the compact pass)
    long long npx;
    float inv_w[UV_NH];
    int W;
    bool vec;                    // W % 4 == 0: a lane's 4 pixels are one aligned float4 per plane
    bool hue_plane;              // opponent mapper: plane 2 = hue (the map pass will read the planes)
    __device__ __forceinline__ void operator()(int y, int gx, const float (&v)[4][3], bool ok) {
        if (!ok || gx >= W) return;
        // planes written: the histogrammed quantities, and for the opponent mapper its hue as well -- the map pass then
        // is a plain element-wise kernel on (radius, L, hue) instead of a second walk (decode, adaptation, blur, atan2)
        constexpr int NPL = QS == QS_OPP ? 3 : QCount<QS>::value;
        float q[4][UV_NH];
        const bool full = gx + 3 < W;             // every lane but the one on the frame's right edge: no per-pixel bound checks
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            quantities<QS>(v[j], q[j]);
            if (QS == QS_OPP && hue_plane) q[j][2] = opp_hue<false>(v[j]);
        }
        if (full) {
#pragma unroll
            for (int j = 0; j < 4; ++j)
#pragma unroll
                for (int h = 0; h < QCount<QS>::value; ++h) atomicAdd(&hs[h * UV_BINS + bin_of(q[j][h], inv_w[h])], 1u);
        } else {
#pragma unroll
            for (int j = 0; j < 4; ++j)
                if (gx + j < W) {
#pragma unroll
                    for (int h = 0; h < QCount<QS>::value; ++h) atomicAdd(&hs[h * UV_BINS + bin_of(q[j][h], inv_w[h])], 1u);
                }
        }
        const long long o = (long long)y * W + gx;
#pragma unroll
        for (int h = 0; h < NPL; ++h) {
            if (h >= QCount<QS>::value && !hue_plane) break;
            float *d = planes + h * npx + o;
            if (vec) {
                *reinterpret_cast<float4 *>(d) = make_float4(q[0][h], q[1][h], q[2][h], q[3][h]);
            } else {
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    if (gx + j < W) d[j] = q[j][h];
            }
        }
    }
};

template <int QS, int R, bool BANDS>
__global__ void __launch_bounds__(UV_THREADS, UV_MINB) uv_hist_kernel(const __grid_constant__ UvParams p) {
    __shared__ float lut_s[256];
    __shared__ uint32_t hs[QCount<QS>::value * UV_BINS];
    const int tid = threadIdx.x, frame = blockIdx.y;
    for (int i = tid; i < 256; i += UV_THREADS) lut_s[i] = __ldg(p.lut + i);
    for (int i = tid; i < QCount<QS>::value * UV_BINS; i += UV_THREADS) hs[i] = 0u;
    __syncthreads();
    const UvFrameStats &st = p.stats[frame];
    Catcher<BANDS> cat;
    cat.init_adapted(p, st, lut_s);
    HistOp<QS> op;
    op.hs = hs;
    op.npx = (long long)p.io.H * p.io.W;
    op.planes = p.planes + (long long)frame * UV_NH * op.npx;
    op.vec = (p.io.W & 3) == 0;
    op.hue_plane = map_from_planes(p);
#pragma unroll
    for (int h = 0; h < UV_NH; ++h) op.inv_w[h] = st.inv_w[h];
    op.W = p.io.W;
    const uint8_t *src = p.io.in + (int64_t)frame * p.io.in_fs;
    const int tasks = p.strips_x * p.strips_y;
    for (int task = blockIdx.x * UV_WARPS + (tid >> 5); task < tasks; task += gridDim.x * UV_WARPS) {
        int xs, ys, rows;
        strip_of<R>(p, task, xs, ys, rows);
        uv_walk<R>(p, cat, src, xs, ys, rows, op);
    }
    __syncthreads();
    uint32_t *gh = p.hist + (int64_t)frame * UV_NH * UV_BINS;
    for (int i = tid; i < QCount<QS>::value * UV_BINS; i += UV_THREADS) {
        const uint32_t c = hs[i];
        if (c) atomicAdd(gh + i, c);
    }
}

// ------------------------------------------------------------------ scan: counts -> candidate bins
__global__ void __launch_bounds__(256) uv_scan_kernel(const __grid_constant__ UvParams p) {
    const int frame = blockIdx.x, tid = threadIdx.x;
    UvFrameStats &st = p.stats[frame];
    __shared__ uint32_t part[256];
    __shared__ uint32_t res[4];      // bin_lo, below_lo, bin_hi, unused
    constexpr int PER = UV_BINS / 256;
    for (int r = 0; r < p.n_req; ++r) {
        const uint32_t *h = p.hist + ((int64_t)frame * UV_NH + p.req_hist[r]) * UV_BINS;
        const uint32_t k_lo = (uint32_t)p.k_lo[r], k_hi = (uint32_t)p.k_hi[r];
        uint32_t loc[PER], s = 0;
#pragma unroll
        for (int j = 0; j < PER; ++j) { loc[j] = h[tid * PER + j]; s += loc[j]; }
        part[tid] = s;
        __syncthreads();
        if (tid == 0) {
            uint32_t run = 0;
            for (int i = 0; i < 256; ++i) { const uint32_t v = part[i]; part[i] = run; run += v; }
        }
        __syncthreads();
        uint32_t run = part[tid];
#pragma unroll
        for (int j = 0; j < PER; ++j) {
            if (k_lo >= run && k_lo < run + loc[j]) { res[0] = tid * PER + j; res[1] = run; }
            if (k_hi >= run && k_hi < run + loc[j]) res[2] = tid * PER + j;
            run += loc[j];
        }
        __syncthreads();
        if (tid == 0) {
            st.bin_lo[r] = res[0];
            st.bin_hi[r] = res[2];
            st.rank_lo[r] = k_lo - res[1];
            st.rank_hi[r] = k_hi - res[1];
            st.cand_count[r] = 0u;
        }
        __syncthreads();
    }
}

// ------------------------------------------------------------------ compact
// Reads the quantity planes the hist pass wrote (4 B per pixel and quantity instead of recomputing
// catches + blur + mapper quantities) and appends every value whose bin is one of the request's
// candidate bins to the request's list -- warp-aggregated, one atomic per warp and hit.
constexpr int CP_PER_THREAD = 16, CP_PER_BLOCK = 256 * CP_PER_THREAD;
__global__ void __launch_bounds__(256) uv_compact_kernel(const __grid_constant__ UvParams p) {
    const int r = blockIdx.y, frame = blockIdx.z, lane = threadIdx.x & 31;
    UvFrameStats &st = p.stats[frame];
    const long long npx = (long long)p.io.H * p.io.W;
    const int h = p.req_hist[r];
    const float inv_w = st.inv_w[h];
    const int lo = (int)st.bin_lo[r], hi = (int)st.bin_hi[r];
    const float *src = p.planes + ((long long)frame * UV_NH + h) * npx;
    float *dst = p.cand + ((long long)frame * p.n_req + r) * p.cap;
    // thread t of the block owns pixels base + 4*(t + 256*k) .. +3, k = 0..3: four independent
    // 16-byte loads in flight per thread, coalesced across the warp
    const long long base = (long long)blockIdx.x * CP_PER_BLOCK;
    float v[CP_PER_THREAD];
    unsigned hits = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const long long i = base + 4 * (threadIdx.x + 256 * k);
        if (i + 3 < npx && (npx & 3) == 0) {
            const float4 t = __ldg(reinterpret_cast<const float4 *>(src + i));
            v[4 * k] = t.x; v[4 * k + 1] = t.y; v[4 * k + 2] = t.z; v[4 * k + 3] = t.w;
        } else {
#pragma unroll
            for (int j = 0; j < 4; ++j) v[4 * k + j] = (i + j < npx) ? __ldg(src + i + j) : -1.f;
        }
    }
#pragma unroll
    for (int e = 0; e < CP_PER_THREAD; ++e) {
        const int b = bin_of(v[e], inv_w);
        if (v[e] >= 0.f && b >= lo && b <= hi) hits |= 1u << e;      // v < 0 marks "past the end"
    }
    if (!__any_sync(FULL, hits != 0)) return;
#pragma unroll
    for (int e = 0; e < CP_PER_THREAD; ++e) {
        const bool hit = (hits >> e) & 1u;
        const unsigned m = __ballot_sync(FULL, hit);
        if (m) {
            const int leader = __ffs(m) - 1;
            uint32_t off = 0;
            if (lane == leader) off = atomicAdd(&st.cand_count[r], (uint32_t)__popc(m));
            off = __shfl_sync(FULL, off, leader);
            if (hit) dst[off + __popc(m & ((1u << lane) - 1u))] = v[e] + 0.f;
        }
    }
}

// ------------------------------------------------------------------ select: exact order statistics
// One CTA per (request, frame): three-level radix select (11 + 11 + 10 bits of the non-negative
// float patterns) for the lower order statistic, one more sweep for the upper one, then the linear
// interpolation numpy.percentile does.
constexpr int SEL_THREADS = 1024;

__device__ __forceinline__ void sel_find(const uint32_t *h, int nbins, uint32_t rank, uint32_t *scratch, uint32_t *out /*bin, rem*/) {
    // h: smem histogram (nbins <= 2048); every thread owns 2 bins; block-wide exclusive scan
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const uint32_t a = (2 * tid < nbins) ? h[2 * tid] : 0u, b = (2 * tid + 1 < nbins) ? h[2 * tid + 1] : 0u;
    uint32_t s = a + b, inc = s;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_up_sync(FULL, inc, o);
        if (lane >= o) inc += t;
    }
    if (lane == 31) scratch[wid] = inc;
    __syncthreads();
    if (wid == 0) {
        uint32_t v = scratch[lane], iv = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t t = __shfl_up_sync(FULL, iv, o);
            if (lane >= o) iv += t;
        }
        scratch[lane] = iv - v;          // exclusive warp offsets
    }
    __syncthreads();
    const uint32_t run = scratch[wid] + inc - s;
    if (rank >= run && rank < run + a) { out[0] = 2 * tid; out[1] = rank - run; }
    else if (rank >= run + a && rank < run + s) { out[0] = 2 * tid + 1; out[1] = rank - run - a; }
    __syncthreads();
}

__global__ void __launch_bounds__(SEL_THREADS) uv_select_kernel(const __grid_constant__ UvParams p) {
    const int r = blockIdx.x, frame = blockIdx.y, tid = threadIdx.x;
    UvFrameStats &st = p.stats[frame];
    __shared__ uint32_t h[UV_BINS];
    __shared__ uint32_t scratch[32];
    __shared__ uint32_t found[2];
    __shared__ uint32_t cnt_le, min_gt;
    const uint32_t cnt = st.cand_count[r];
    const uint32_t *vals = reinterpret_cast<const uint32_t *>(p.cand + ((long long)frame * p.n_req + r) * p.cap);
    uint32_t rank = st.rank_lo[r];
    uint32_t prefix = 0;
    const int shifts[3] = {21, 10, 0}, nbits[3] = {11, 11, 10};
    for (int lv = 0; lv < 3; ++lv) {
        for (int i = tid; i < UV_BINS; i += SEL_THREADS) h[i] = 0u;
        __syncthreads();
        const int sh = shifts[lv], nb = nbits[lv];
        const uint32_t mask = (1u << nb) - 1u;
        for (uint32_t i = tid; i < cnt; i += SEL_THREADS) {
            const uint32_t b = vals[i];
            if (lv == 0 || (b >> (sh + nb)) == prefix) atomicAdd(&h[(b >> sh) & mask], 1u);
        }
        __syncthreads();
        sel_find(h, 1 << nb, rank, scratch, found);
        prefix = (prefix << nb) | found[0];
        rank = found[1];
        __syncthreads();
    }
    const uint32_t a_bits = prefix;
    if (tid == 0) { cnt_le = 0u; min_gt = 0xffffffffu; }
    __syncthreads();
    uint32_t le = 0, mg = 0xffffffffu;
    for (uint32_t i = tid; i < cnt; i += SEL_THREADS) {
        const uint32_t b = vals[i];
        if (b <= a_bits) ++le; else mg = min(mg, b);
    }
    atomicAdd(&cnt_le, le);
    atomicMin(&min_gt, mg);
    __syncthreads();
    if (tid == 0) {
        uint32_t b_bits = a_bits;
        if (st.rank_hi[r] >= cnt_le && min_gt != 0xffffffffu) b_bits = min_gt;
        st.pct[r] = numpy_lerp(__uint_as_float(a_bits), __uint_as_float(b_bits), p.gamma[r]);
    }
}

// ------------------------------------------------------------------ map
struct MapConsts {
    float pr, pL, rpr, rpL;       // opponent: percentile + eps, and reciprocals
    float d95[3], d98;            // falsecolor / purple: max(percentile, eps)
    float r95[3], r98;            // reciprocals
    float c0[3], c1[3], pd[3];    // purple / warm anchors (linear light, host-computed) and accent direction
    float m[9];
    float alpha;
};

__device__ __forceinline__ void falsecolor(const float (&c)[3], const MapConsts &k, float (&rgb)[3]) {
    // uv_mappers.py:29-43 (python-float coefficients act as float32)
    const float Un = div_by(c[0], k.d95[0], k.r95[0]), Bn = div_by(c[1], k.d95[1], k.r95[1]), Gn = div_by(c[2], k.d95[2], k.r95[2]);
    rgb[0] = __saturatef(__fadd_rn(__fmul_rn(0.85f, Un), __fmul_rn(0.10f, Gn)));
    rgb[1] = __saturatef(__fadd_rn(__fmul_rn(0.80f, Gn), __fmul_rn(0.20f, Bn)));
    rgb[2] = __saturatef(__fadd_rn(__fmul_rn(0.70f, Bn), __fmul_rn(0.40f, Un)));
}

__device__ __forceinline__ void purple_soft(float U, const MapConsts &k, float (&rgb)[3]) {
    // uv_mappers.py:90-132 with the defaults u_gamma .90, accent_gamma .85, accent_strength .05
    const float u = powf(__saturatef(div_by(U, k.d98, k.r98)), 0.90f);
    const float w = powf(u, 0.85f);
    float y = 0.f;
    const float yc[3] = {0.2126f, 0.7152f, 0.0722f};
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        float v = __fadd_rn(__fmul_rn(__fsub_rn(1.0f, u), k.c0[i]), __fmul_rn(u, k.c1[i]));
        v = __fadd_rn(v, __fmul_rn(__fmul_rn(0.05f, w), k.pd[i]));
        rgb[i] = v;
    }
    y = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(yc[0], rgb[0]), __fmul_rn(yc[1], rgb[1])), __fmul_rn(yc[2], rgb[2])), 1e-8f);
    const float yt = __saturatef(__fadd_rn(0.22f, __fmul_rn(0.55f, u)));
    const float gain = fminf(fmaxf(__fdiv_rn(yt, y), 0.6f), 1.6f);
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        const float v = __fmul_rn(rgb[i], gain);
        rgb[i] = __saturatef(__fdiv_rn(v, __fadd_rn(1.0f, __fmul_rn(0.6f, v))));
    }
}

// hsv_to_rgb (uv_mappers.py:14-26) of hue, sat = clip(radius / (P99 + eps)), val = clip(L / (P99 + eps)).
// Channel c = val * (1 - sat * m_c), m_c = clamp(min(k, 4 - k), 0, 1), k = (n_c + 6 hue) mod 6, n = (5, 3, 1): m is exactly
// 0, 1, f or 1 - f in every sextant, so these are the p / q / t products of the reference's np.select without a branch
// (NumPy evaluates q and t in float64 and rounds once; one fused multiply-add keeps the float32 evaluation within an ulp of
// that).  Measured, 20 4K frames: 1.178 ms against 1.240 ms for a divergent switch over the sextant.
__device__ __forceinline__ void opp_color(float radius, float L, float hue, const MapConsts &k, float (&rgb)[3]) {
    const float sat = __saturatef(div_by(radius, k.pr, k.rpr));
    const float val = __saturatef(div_by(L, k.pL, k.rpL));
    const float h6 = __fmul_rn(hue, 6.0f);
    const float hh = h6 >= 6.0f ? h6 - 6.0f : h6;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        float kk = hh + (float)(5 - 2 * c);
        kk = kk >= 6.0f ? kk - 6.0f : kk;
        const float m = __saturatef(fminf(kk, 4.0f - kk));
        rgb[c] = __fmul_rn(val, fmaf(-m, sat, 1.0f));
    }
}

template <int MAPPER, bool PRECISE = false>
__device__ __forceinline__ void map_pixel(const float (&c)[3], const MapConsts &k, float (&rgb)[3]) {
    if (MAPPER == MAP_OPPONENT) {
        // uv_mappers.py:53-64 and hsv_to_rgb :14-26
        float q[UV_NH];
        quantities<QS_OPP, PRECISE>(c, q);
        opp_color(q[0], q[1], opp_hue<PRECISE>(c), k, rgb);
    } else if (MAPPER == MAP_FALSECOLOR) {
        falsecolor(c, k, rgb);
    } else if (MAPPER == MAP_MATRIX) {
        // uv_mappers.py:45-50: [U,B,G] @ M.T
#pragma unroll
        for (int i = 0; i < 3; ++i) rgb[i] = k.m[3 * i] * c[0] + k.m[3 * i + 1] * c[1] + k.m[3 * i + 2] * c[2];
    } else if (MAPPER == MAP_PURPLE) {
        purple_soft(c[0], k, rgb);
    } else {
        // uv_mappers.py:135-144; the trailing P99 normalisation divides by max(1, p99) and every
        // mixed value is <= 1, so it is the identity
        float a[3], b[3];
        falsecolor(c, k, a);
        purple_soft(c[0], k, b);
#pragma unroll
        for (int i = 0; i < 3; ++i) rgb[i] = __fadd_rn(__fmul_rn(__fsub_rn(1.0f, k.alpha), a[i]), __fmul_rn(k.alpha, b[i]));
    }
}

template <int MAPPER>
struct MapOp {
    MapConsts k;
    EncTable enc;
    uint8_t *dst;
    int64_t out_rs;
    int W;
    bool aligned;
    __device__ __forceinline__ void operator()(int y, int gx, const float (&v)[4][3], bool ok) {
        if (!ok || gx >= W) return;
        uint32_t by[12];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            float rgb[3];
            map_pixel<MAPPER>(v[j], k, rgb);
#pragma unroll
            for (int i = 0; i < 3; ++i) by[3 * j + i] = encode_u8(enc, rgb[i]);
        }
        uint8_t *o = dst + (int64_t)y * out_rs + 3 * gx;
        if (aligned && gx + 3 < W) {
            uint32_t *o32 = reinterpret_cast<uint32_t *>(o);
#pragma unroll
            for (int q = 0; q < 3; ++q) o32[q] = by[4 * q] | (by[4 * q + 1] << 8) | (by[4 * q + 2] << 16) | (by[4 * q + 3] << 24);
        } else {
            const int nb = 3 * min(4, W - gx);
#pragma unroll
            for (int q = 0; q < 12; ++q)
                if (q < nb) o[q] = (uint8_t)by[q];
        }
    }
};

template <int MAPPER, int R, bool BANDS>
__global__ void __launch_bounds__(UV_THREADS, UV_MINB) uv_map_kernel(const __grid_constant__ UvParams p) {
    __shared__ float lut_s[256];
    __shared__ uint32_t enc_s[AVB_ENC_TABLE_MAX];
    const int tid = threadIdx.x, frame = blockIdx.y;
    for (int i = tid; i < 256; i += UV_THREADS) lut_s[i] = __ldg(p.lut + i);
    copy_to_smem(enc_s, p.enc, min((int)AVB_ENC_TABLE_MAX, ENC_HEADER + (int)__ldg(p.enc + 2)));
    __syncthreads();
    const UvFrameStats &st = p.stats[frame];
    Catcher<BANDS> cat;
    cat.init_adapted(p, st, lut_s);
    MapOp<MAPPER> op;
    op.enc = enc_view(enc_s);
    op.dst = p.io.out + (int64_t)frame * p.io.out_fs;
    op.out_rs = p.io.out_rs;
    op.W = p.io.W;
    op.aligned = p.aligned_out != 0;
    MapConsts &k = op.k;
    k.pr = st.pct[0] + p.eps;               // uv_mappers.py:61-62: percentile + eps, float32
    k.pL = st.pct[1] + p.eps;
    k.rpr = __frcp_rn(k.pr);
    k.rpL = __frcp_rn(k.pL);
#pragma unroll
    for (int i = 0; i < 3; ++i) { k.d95[i] = fmaxf(st.pct[i], p.eps); k.r95[i] = __frcp_rn(k.d95[i]); }
    k.d98 = fmaxf(MAPPER == MAP_PURPLE ? st.pct[0] : st.pct[3], p.eps);
    k.r98 = __frcp_rn(k.d98);
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        k.c0[i] = p.anchors[i];
        k.c1[i] = p.anchors[3 + i];
        k.pd[i] = __fsub_rn(k.c0[i], 0.5f);
        k.m[3 * i] = p.map_m[3 * i]; k.m[3 * i + 1] = p.map_m[3 * i + 1]; k.m[3 * i + 2] = p.map_m[3 * i + 2];
    }
    k.alpha = p.mix_alpha;
    const uint8_t *src = p.io.in + (int64_t)frame * p.io.in_fs;
    const int tasks = p.strips_x * p.strips_y;
    for (int task = blockIdx.x * UV_WARPS + (tid >> 5); task < tasks; task += gridDim.x * UV_WARPS) {
        int xs, ys, rows;
        strip_of<R>(p, task, xs, ys, rows);
        uv_walk<R>(p, cat, src, xs, ys, rows, op);
    }
}


__device__ __forceinline__ void fill_map_consts(const UvParams &p, const UvFrameStats &st, int mapper, MapConsts &k) {
    k.pr = st.pct[0] + p.eps;               // uv_mappers.py:61-62: percentile + eps, float32
    k.pL = st.pct[1] + p.eps;
    k.rpr = __frcp_rn(k.pr);
    k.rpL = __frcp_rn(k.pL);
#pragma unroll
    for (int i = 0; i < 3; ++i) { k.d95[i] = fmaxf(st.pct[i], p.eps); k.r95[i] = __frcp_rn(k.d95[i]); }
    k.d98 = fmaxf(mapper == MAP_PURPLE ? st.pct[0] : st.pct[3], p.eps);
    k.r98 = __frcp_rn(k.d98);
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        k.c0[i] = p.anchors[i];
        k.c1[i] = p.anchors[3 + i];
        k.pd[i] = __fsub_rn(k.c0[i], 0.5f);
        k.m[3 * i] = p.map_m[3 * i]; k.m[3 * i + 1] = p.map_m[3 * i + 1]; k.m[3 * i + 2] = p.map_m[3 * i + 2];
    }
    k.alpha = p.mix_alpha;
}

// ------------------------------------------------------------------ map pass on the hist pass's planes
// Opponent mapper: (radius, L, hue) -> hsv_to_rgb -> sRGB encode; the other mappers: (U, B, G) -> map_pixel -> encode: element-wise, four pixels per thread (one float4 per plane in, three
// 32-bit words out).  Same functions, same operands as the walk (the planes hold exactly the values the walk recomputes),
// so the bytes are identical; what disappears is the second decode + adaptation + blur + atan2 per pixel
// (215 -> ~60 instructions per pixel) at the price of 12 instead of 3 bytes read per pixel -- the path is issue bound.
constexpr int MP_THREADS = 256, MP_GROUPS = 4;       // groups of four pixels per thread
#ifndef MP_MINB
#define MP_MINB 4        // measured: 3 -> 0.578 ms, 4 -> 0.554 ms per 20 4K frames
#endif
template <int MAPPER>
__global__ void __launch_bounds__(MP_THREADS, MP_MINB) uv_map_planes_kernel(const __grid_constant__ UvParams p) {
    constexpr int NPL = MAPPER == MAP_PURPLE ? 1 : 3;       // planes the hist pass wrote for this mapper
    __shared__ uint32_t enc_s[AVB_ENC_TABLE_MAX];
    const int tid = threadIdx.x, frame = blockIdx.y;
    copy_to_smem(enc_s, p.enc, min((int)AVB_ENC_TABLE_MAX, ENC_HEADER + (int)__ldg(p.enc + 2)));
    __syncthreads();
    const EncTable enc = enc_view(enc_s);
    const UvFrameStats &st = p.stats[frame];
    MapConsts k;
    fill_map_consts(p, st, MAPPER, k);
    const int W = p.io.W;
    const uint32_t W4 = (uint32_t)W >> 2;
    const long long npx = (long long)p.io.H * W;
    const uint32_t groups = (uint32_t)(npx >> 2);    // < 2^31: a frame of 2^33 pixels does not exist
    const float *pl = p.planes + (long long)frame * UV_NH * npx;
    uint8_t *dst = p.io.out + (int64_t)frame * p.io.out_fs;
    const uint32_t g0 = (blockIdx.x * MP_GROUPS) * MP_THREADS + tid;
    float4 qr[MP_GROUPS], qL[MP_GROUPS], qh[MP_GROUPS];
#pragma unroll
    for (int u = 0; u < MP_GROUPS; ++u) {            // all loads first: twelve 16-byte requests in flight per thread
        const uint32_t g = g0 + (uint32_t)u * MP_THREADS;
        if (g < groups) {
            qr[u] = __ldcs(reinterpret_cast<const float4 *>(pl) + g);
            if (NPL > 1) {
                qL[u] = __ldcs(reinterpret_cast<const float4 *>(pl + npx) + g);
                qh[u] = __ldcs(reinterpret_cast<const float4 *>(pl + 2 * npx) + g);
            } else {
                qL[u] = qh[u] = make_float4(0.f, 0.f, 0.f, 0.f);
            }
        }
    }
    // (row, group in the row) of the first group by one 32-bit division, of the following ones by stepping
    uint32_t y = g0 / W4, x4 = g0 - y * W4;
#pragma unroll
    for (int u = 0; u < MP_GROUPS; ++u) {
        const uint32_t g = g0 + (uint32_t)u * MP_THREADS;
        if (g >= groups) break;
        if (u > 0) {
            x4 += MP_THREADS;
            while (x4 >= W4) { x4 -= W4; ++y; }
        }
        const float r4[4] = {qr[u].x, qr[u].y, qr[u].z, qr[u].w}, L4[4] = {qL[u].x, qL[u].y, qL[u].z, qL[u].w};
        const float h4[4] = {qh[u].x, qh[u].y, qh[u].z, qh[u].w};
        uint32_t by[12];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            float rgb[3];
            if (MAPPER == MAP_OPPONENT) {
                opp_color(r4[j], L4[j], h4[j], k, rgb);
            } else {
                const float c[3] = {r4[j], L4[j], h4[j]};          // the catches (U, B, G); the purple map reads U only
                map_pixel<MAPPER>(c, k, rgb);
            }
#pragma unroll
            for (int i = 0; i < 3; ++i) by[3 * j + i] = encode_u8(enc, rgb[i]);
        }
        uint32_t *o32 = reinterpret_cast<uint32_t *>(dst + (int64_t)y * p.io.out_rs + 12u * x4);
#pragma unroll
        for (int q = 0; q < 3; ++q) o32[q] = by[4 * q] | (by[4 * q + 1] << 8) | (by[4 * q + 2] << 16) | (by[4 * q + 3] << 24);
    }
}

// ------------------------------------------------------------------ float32 plane path
// The generality route (float / wide-integer frames, hsi_downsample, blur radii beyond the fused walker):
// the (U,B,G) planes live in HBM as packed float32 [n,H,W,3] and are produced by k6_imgops steps; these
// kernels are the same mapper / percentile code as above on a plain grid-stride pixel loop.
__device__ __forceinline__ float srgb_decode_torch(float t) {      // classic_rgb_to_hsi.py:16-22, float32 like torch
    return t <= 0.04045f ? __fdiv_rn(t, 12.92f) : powf(__fdiv_rn(t + 0.055f, 1.055f), 2.4f);
}
__device__ __forceinline__ float srgb_encode_uv(float l) {         // uv_helpers.py:40-44 (1/2.4 acts as a float32 scalar)
    return l <= 0.0031308f ? __fmul_rn(l, 12.92f) : __fsub_rn(__fmul_rn(1.055f, powf(fmaxf(l, 0.f), 0.41666666f)), 0.055f);
}

struct CatchF32P {
    const float *in; float *out; long long npx;      // img01 -> raw catches, both packed x3
    UvParams uv;
};
template <bool BANDS>
__global__ void __launch_bounds__(256) uv_catches_f32_kernel(const __grid_constant__ CatchF32P p) {
    Catcher<BANDS> cat;
    cat.init_raw(p.uv, nullptr);
    for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < p.npx; i += (long long)gridDim.x * 256) {
        const float c0 = srgb_decode_torch(p.in[3 * i]), c1 = srgb_decode_torch(p.in[3 * i + 1]), c2 = srgb_decode_torch(p.in[3 * i + 2]);
        float u, b, g;
        cat.from_linear(c0, c1, c2, u, b, g);
        p.out[3 * i] = u; p.out[3 * i + 1] = b; p.out[3 * i + 2] = g;
    }
}

struct PlaneP {
    const float *ubg;           // [n][H*W][3] adapted + blurred catches
    void *out;                  // uint8 (strided frames) or float32 packed
    int out_f32, quantize;
    UvParams uv;
};

// per-frame channel maxima of the planes -> UvFrameStats.max_bits (bin sizing only)
__global__ void __launch_bounds__(256) uv_planemax_kernel(const __grid_constant__ PlaneP p) {
    const int frame = blockIdx.y;
    const long long npx = (long long)p.uv.io.H * p.uv.io.W;
    const float *f = p.ubg + (long long)frame * npx * 3;
    float m[3] = {0.f, 0.f, 0.f};
    for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < npx; i += (long long)gridDim.x * 256) {
#pragma unroll
        for (int k = 0; k < 3; ++k) m[k] = fmaxf(m[k], f[3 * i + k]);
    }
#pragma unroll
    for (int k = 0; k < 3; ++k) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) m[k] = fmaxf(m[k], __shfl_xor_sync(FULL, m[k], o));
        if ((threadIdx.x & 31) == 0) atomicMax(&p.uv.stats[frame].max_bits[k], __float_as_uint(m[k]));
    }
}

template <int QS>
__global__ void __launch_bounds__(256) uv_hist_f32_kernel(const __grid_constant__ PlaneP p) {
    __shared__ uint32_t hs[QCount<QS>::value * UV_BINS];
    const int tid = threadIdx.x, frame = blockIdx.y;
    for (int i = tid; i < QCount<QS>::value * UV_BINS; i += 256) hs[i] = 0u;
    __syncthreads();
    const UvFrameStats &st = p.uv.stats[frame];
    const long long npx = (long long)p.uv.io.H * p.uv.io.W;
    const float *f = p.ubg + (long long)frame * npx * 3;
    float *planes = p.uv.planes + (long long)frame * UV_NH * npx;
    for (long long i = (long long)blockIdx.x * 256 + tid; i < npx; i += (long long)gridDim.x * 256) {
        const float c[3] = {f[3 * i], f[3 * i + 1], f[3 * i + 2]};
        float q[UV_NH];
        quantities<QS, true>(c, q);
#pragma unroll
        for (int h = 0; h < QCount<QS>::value; ++h) {
            // catches are non-negative by construction (non-negative lobes, illuminant, sensitivities, blur and
            // area / linear resampling weights), as on the uint8 route
            atomicAdd(&hs[h * UV_BINS + bin_of(q[h], st.inv_w[h])], 1u);
            planes[h * npx + i] = q[h];
        }
    }
    __syncthreads();
    uint32_t *gh = p.uv.hist + (int64_t)frame * UV_NH * UV_BINS;
    for (int i = tid; i < QCount<QS>::value * UV_BINS; i += 256)
        if (hs[i]) atomicAdd(gh + i, hs[i]);
}

template <int MAPPER>
__global__ void __launch_bounds__(256) uv_map_f32_kernel(const __grid_constant__ PlaneP p) {
    __shared__ uint32_t enc_s[AVB_ENC_TABLE_MAX];
    const int frame = blockIdx.y;
    if (!p.out_f32) copy_to_smem(enc_s, p.uv.enc, min((int)AVB_ENC_TABLE_MAX, ENC_HEADER + (int)__ldg(p.uv.enc + 2)));
    __syncthreads();
    const EncTable enc = enc_view(enc_s);
    MapConsts k;
    fill_map_consts(p.uv, p.uv.stats[frame], MAPPER, k);
    const int W = p.uv.io.W;
    const long long npx = (long long)p.uv.io.H * W;
    const float *f = p.ubg + (long long)frame * npx * 3;
    for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < npx; i += (long long)gridDim.x * 256) {
        const float c[3] = {f[3 * i], f[3 * i + 1], f[3 * i + 2]};
        float rgb[3];
        map_pixel<MAPPER, true>(c, k, rgb);
        if (p.out_f32) {
            float *o = static_cast<float *>(p.out) + ((long long)frame * npx + i) * 3;
#pragma unroll
            for (int ch = 0; ch < 3; ++ch) {
                float v = srgb_encode_uv(__saturatef(rgb[ch]));        // honeybee.py:166-169
                if (p.quantize) v = truncf(__fadd_rn(__fmul_rn(v, 255.0f), 0.5f));       // :170-171 for integer dtypes
                o[ch] = v;
            }
        } else {
            const int y = (int)(i / W), x = (int)(i - (long long)y * W);
            uint8_t *o = static_cast<uint8_t *>(p.out) + (int64_t)frame * p.uv.io.out_fs + (int64_t)y * p.uv.io.out_rs + 3 * x;
#pragma unroll
            for (int ch = 0; ch < 3; ++ch) o[ch] = (uint8_t)encode_u8(enc, rgb[ch]);
        }
    }
}

template <int MAPPER>
static int launch_mapper_f32(const PlaneP &pp, cudaStream_t st) {
    constexpr int QS = MAPPER == MAP_OPPONENT ? QS_OPP : (MAPPER == MAP_PURPLE ? QS_U : QS_UBG);
    const UvParams &p = pp.uv;
    const long long npx = (long long)p.io.H * p.io.W;
    const unsigned bx = (unsigned)std::max<long long>(1, std::min<long long>((npx + 255) / 256, (long long)sm_count() * 8 / p.io.n + 1));
    if (p.n_req > 0) {
        {
            AVB_TIMED("k3_uv_planemax", st);
            uv_planemax_kernel<<<dim3(bx, p.io.n), 256, 0, st>>>(pp);
        }
        {
            AVB_TIMED("k3_uv_prep", st);
            uv_prep_kernel<QS><<<(p.io.n + 63) / 64, 64, 0, st>>>(p);      // adapt = 0: bins sized from the plane maxima
        }
        {
            AVB_TIMED("k3_uv_hist_f32", st);
            uv_hist_f32_kernel<QS><<<dim3(bx, p.io.n), 256, 0, st>>>(pp);
        }
        {
            AVB_TIMED("k3_uv_scan", st);
            uv_scan_kernel<<<p.io.n, 256, 0, st>>>(p);
        }
        {
            AVB_TIMED("k3_uv_compact", st);
            uv_compact_kernel<<<dim3((unsigned)((npx + CP_PER_BLOCK - 1) / CP_PER_BLOCK), p.n_req, p.io.n), 256, 0, st>>>(p);
        }
        {
            AVB_TIMED("k3_uv_select", st);
            uv_select_kernel<<<dim3(p.n_req, p.io.n), SEL_THREADS, 0, st>>>(p);
        }
    }
    {
        AVB_TIMED("k3_uv_map_f32", st);
        uv_map_f32_kernel<MAPPER><<<dim3(bx, p.io.n), 256, 0, st>>>(pp);
    }
    AVB_CUDA_OK(cudaGetLastError());
    return AVB_OK;
}

// ------------------------------------------------------------------ launch plumbing
static int qset_of(int mapper) {
    switch (mapper) {
        case MAP_OPPONENT: return QS_OPP;
        case MAP_PURPLE: return QS_U;
        default: return QS_UBG;
    }
}

static dim3 walk_grid(const UvParams &p, int per_sm) {
    const int tasks = p.strips_x * p.strips_y;
    int bx = (tasks + UV_WARPS - 1) / UV_WARPS;
    const int cap = sm_count() * per_sm / p.io.n;          // rounded DOWN: one CTA too many per frame costs a whole second wave
    if (bx > cap) bx = cap < 1 ? 1 : cap;
    return dim3(bx, p.io.n);
}

template <int QS, int R, bool BANDS>
static int launch_percentiles(const UvParams &p, cudaStream_t st) {
    {
        AVB_TIMED("k3_uv_hist", st);
        uv_hist_kernel<QS, R, BANDS><<<walk_grid(p, 4 * UV_HIST_WAVES), UV_THREADS, 0, st>>>(p);
    }
    {
        AVB_TIMED("k3_uv_scan", st);
        uv_scan_kernel<<<p.io.n, 256, 0, st>>>(p);
    }
    {
        AVB_TIMED("k3_uv_compact", st);
        const long long npx = (long long)p.io.H * p.io.W;
        uv_compact_kernel<<<dim3((unsigned)((npx + CP_PER_BLOCK - 1) / CP_PER_BLOCK), p.n_req, p.io.n), 256, 0, st>>>(p);
    }
    {
        AVB_TIMED("k3_uv_select", st);
        uv_select_kernel<<<dim3(p.n_req, p.io.n), SEL_THREADS, 0, st>>>(p);
    }
    AVB_CUDA_OK(cudaGetLastError());
    return AVB_OK;
}

template <int MAPPER, int R, bool BANDS>
static int launch_mapper(const UvParams &p, cudaStream_t st) {
    constexpr int QS = MAPPER == MAP_OPPONENT ? QS_OPP : (MAPPER == MAP_PURPLE ? QS_U : QS_UBG);
    {
        AVB_TIMED("k3_uv_prep", st);
        uv_prep_kernel<QS><<<(p.io.n + 63) / 64, 64, 0, st>>>(p);
    }
    if (p.n_req > 0)
        if (int e = launch_percentiles<QS, R, BANDS>(p, st)) return e;
    if (MAPPER != MAP_MATRIX && map_from_planes(p)) {
        AVB_TIMED("k3_uv_map", st);
        const long long groups = ((long long)p.io.H * p.io.W) >> 2, per_cta = (long long)MP_THREADS * MP_GROUPS;
        uv_map_planes_kernel<MAPPER><<<dim3((unsigned)((groups + per_cta - 1) / per_cta), p.io.n), MP_THREADS, 0, st>>>(p);
    } else {
        AVB_TIMED("k3_uv_map", st);
        // one task per warp (measured: a persistent grid, 4-5 tasks per warp, is 15 % slower here)
        const int tasks = p.strips_x * p.strips_y;
        uv_map_kernel<MAPPER, R, BANDS><<<dim3((tasks + UV_WARPS - 1) / UV_WARPS, p.io.n), UV_THREADS, 0, st>>>(p);
    }
    AVB_CUDA_OK(cudaGetLastError());
    return AVB_OK;
}

template <int R, bool BANDS>
static int dispatch_mapper(const UvParams &p, cudaStream_t st) {
    switch (p.mapper) {
        case MAP_OPPONENT: return launch_mapper<MAP_OPPONENT, R, BANDS>(p, st);
        case MAP_FALSECOLOR: return launch_mapper<MAP_FALSECOLOR, R, BANDS>(p, st);
        case MAP_MATRIX: return launch_mapper<MAP_MATRIX, R, BANDS>(p, st);
        case MAP_PURPLE: return launch_mapper<MAP_PURPLE, R, BANDS>(p, st);
        default: return launch_mapper<MAP_MIXED, R, BANDS>(p, st);
    }
}

static int n_requests(int mapper) {
    switch (mapper) {
        case MAP_OPPONENT: return 2;
        case MAP_FALSECOLOR: return 3;
        case MAP_MATRIX: return 0;
        case MAP_PURPLE: return 1;
        default: return 4;
    }
}

static size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

}  // namespace avb

using namespace avb;

extern "C" int64_t avb_uv_workspace_bytes(int n, int H, int W, int map_mode) {
    if (n <= 0 || H <= 0 || W <= 0 || map_mode < 0 || map_mode > MAP_MIXED) return 0;
    const size_t stats = align_up((size_t)n * sizeof(UvFrameStats), 256);
    const size_t hist = (size_t)n * UV_NH * UV_BINS * sizeof(uint32_t);
    const size_t planes = n_requests(map_mode) ? (size_t)n * UV_NH * (size_t)H * W * sizeof(float) : 0;
    const size_t cand = (size_t)n * n_requests(map_mode) * (size_t)H * W * sizeof(float);
    return (int64_t)(stats + hist + planes + cand);
}

extern "C" int avb_uv_map_u8(const uint8_t *in, uint8_t *out, int n, int H, int W,
                             int64_t in_frame_stride, int64_t in_row_stride,
                             int64_t out_frame_stride, int64_t out_row_stride,
                             const float *dec_dev, const uint32_t *enc_dev,
                             const float *m3_host, const float *bands_dev, int n_bands, float denom_eps,
                             int adapt_mode, const float *blur_taps_host, int blur_ksize,
                             int map_mode, const float *map_params_host, float mix_alpha,
                             void *workspace_dev, float *dbg_catches_dev, avb_stream_t stream) {
    UvParams p{};
    p.io = FrameIO{in, out, in_frame_stride, in_row_stride, out_frame_stride, out_row_stride, n, H, W};
    AVB_REQUIRE(in && out, "null frame pointer");
    AVB_REQUIRE(n > 0 && H > 0 && W > 0, "bad frame geometry");
    AVB_REQUIRE(n <= 65535, "batch too large for one launch");
    AVB_REQUIRE(in_row_stride >= 3LL * W && out_row_stride >= 3LL * W, "row stride smaller than 3*W");
    AVB_REQUIRE(dec_dev && enc_dev && m3_host && workspace_dev, "null table / workspace pointer");
    AVB_REQUIRE((reinterpret_cast<uintptr_t>(workspace_dev) & 15) == 0, "workspace_dev must be 16-byte aligned (float4 plane accesses)");
    AVB_REQUIRE(n_bands >= 0 && n_bands <= UV_MAX_BANDS && (n_bands == 0 || bands_dev), "bad band table");
    AVB_REQUIRE(adapt_mode >= 0 && adapt_mode <= 2, "adapt_mode must be 0 (none), 1 (white patch) or 2 (gray world)");
    AVB_REQUIRE(blur_ksize == 0 || ((blur_ksize == 3 || blur_ksize == 5) && blur_taps_host), "blur ksize must be 0, 3 or 5");
    AVB_REQUIRE(map_mode >= 0 && map_mode <= MAP_MIXED, "unknown map_mode");
    AVB_REQUIRE(map_mode == MAP_OPPONENT || map_mode == MAP_FALSECOLOR || map_params_host, "this map_mode needs map_params_host");
    AVB_REQUIRE((long long)H * W < (1LL << 31), "frame too large");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    p.lut = dec_dev;
    p.enc = enc_dev;
    for (int i = 0; i < 9; ++i) p.M3[i] = m3_host[i];
    p.bands = bands_dev;
    p.n_bands = n_bands;
    p.denom_eps = denom_eps;
    p.adapt = adapt_mode;
    p.eps = 1e-8f;
    const int R = blur_ksize / 2;
    p.t0 = 1.f; p.t1 = 0.f; p.t2 = 0.f;
    if (R >= 1) { p.t0 = blur_taps_host[R]; p.t1 = blur_taps_host[R + 1]; }
    if (R >= 2) p.t2 = blur_taps_host[R + 2];
    p.mapper = map_mode;
    if (map_params_host) {
        for (int i = 0; i < 9; ++i) p.map_m[i] = map_params_host[i];
        for (int i = 0; i < 6; ++i) p.anchors[i] = map_params_host[9 + i];
    }
    p.mix_alpha = mix_alpha;
    p.dbg_catches = dbg_catches_dev;
    p.aligned_in = ((reinterpret_cast<uintptr_t>(in) | (uintptr_t)in_frame_stride | (uintptr_t)in_row_stride) & 3) == 0;
    p.aligned_out = ((reinterpret_cast<uintptr_t>(out) | (uintptr_t)out_frame_stride | (uintptr_t)out_row_stride) & 3) == 0;
    const int SW = R ? 120 : 128;
    p.strips_x = (W + SW - 1) / SW;
    p.strips_y = (H + UV_RH - 1) / UV_RH;

    // workspace: stats | histograms | candidate lists
    const long long npx = (long long)H * W;
    uint8_t *ws = static_cast<uint8_t *>(workspace_dev);
    const size_t stats_bytes = align_up((size_t)n * sizeof(UvFrameStats), 256);
    const size_t hist_bytes = (size_t)n * UV_NH * UV_BINS * sizeof(uint32_t);
    p.stats = reinterpret_cast<UvFrameStats *>(ws);
    p.hist = reinterpret_cast<uint32_t *>(ws + stats_bytes);
    const size_t planes_bytes = n_requests(map_mode) ? (size_t)n * UV_NH * (size_t)npx * sizeof(float) : 0;
    p.planes = reinterpret_cast<float *>(ws + stats_bytes + hist_bytes);
    p.cand = reinterpret_cast<float *>(ws + stats_bytes + hist_bytes + planes_bytes);
    p.cap = npx;

    // percentile requests (numpy.percentile(method="linear"): virtual index q/100 * (N-1))
    p.n_req = n_requests(map_mode);
    const int qs = qset_of(map_mode);
    const double pcts[5][UV_NR] = {{95, 95, 0, 0}, {95, 95, 95, 0}, {0, 0, 0, 0}, {98, 0, 0, 0}, {95, 95, 95, 98}};
    const int hists[5][UV_NR] = {{0, 1, 0, 0}, {0, 1, 2, 0}, {0, 0, 0, 0}, {0, 0, 0, 0}, {0, 1, 2, 0}};
    (void)qs;
    for (int r = 0; r < p.n_req; ++r) {
        const PctIndex pi = numpy_percentile_index(pcts[map_mode][r], npx);    // float32 virtual index, as NumPy computes it
        p.req_hist[r] = hists[map_mode][r];
        p.k_lo[r] = pi.k_lo; p.k_hi[r] = pi.k_hi; p.gamma[r] = pi.gamma;
    }

    AVB_CUDA_OK(cudaMemsetAsync(ws, 0, stats_bytes + hist_bytes, st));
    {
        int bx = (sm_count() * 16 + n - 1) / n;        // ~16 CTAs per SM over the whole batch
        if (bx > H) bx = H;
        dim3 grid((unsigned)bx, n);
        AVB_TIMED("k3_uv_stats", st);
        if (n_bands) uv_stats_kernel<true><<<grid, 256, 0, st>>>(p);
        else uv_stats_kernel<false><<<grid, 256, 0, st>>>(p);
        AVB_CUDA_OK(cudaGetLastError());
    }
    if (n_bands) {
        switch (R) {
            case 0: return dispatch_mapper<0, true>(p, st);
            case 1: return dispatch_mapper<1, true>(p, st);
            default: return dispatch_mapper<2, true>(p, st);
        }
    }
    switch (R) {
        case 0: return dispatch_mapper<0, false>(p, st);
        case 1: return dispatch_mapper<1, false>(p, st);
        default: return dispatch_mapper<2, false>(p, st);
    }
}

// ---- float32 plane route (include/avb200.h: avb_uv_catches_f32 / avb_uv_map_f32)
extern "C" int avb_uv_catches_f32(const float *img01_dev, float *catches_dev, int64_t npx, const float *m3_host,
                                  const float *bands_dev, int n_bands, float denom_eps, avb_stream_t stream) {
    AVB_REQUIRE(img01_dev && catches_dev && m3_host, "null pointer");
    AVB_REQUIRE(npx > 0, "bad geometry");
    AVB_REQUIRE(n_bands >= 0 && n_bands <= UV_MAX_BANDS && (n_bands == 0 || bands_dev), "bad band table");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    CatchF32P p{};
    p.in = img01_dev; p.out = catches_dev; p.npx = npx;
    for (int i = 0; i < 9; ++i) p.uv.M3[i] = m3_host[i];
    p.uv.bands = bands_dev; p.uv.n_bands = n_bands; p.uv.denom_eps = denom_eps;
    const unsigned bx = (unsigned)std::max<long long>(1, std::min<long long>((npx + 255) / 256, (long long)sm_count() * 16));
    AVB_TIMED("k3_uv_catches_f32", st);
    if (n_bands) uv_catches_f32_kernel<true><<<bx, 256, 0, st>>>(p);
    else uv_catches_f32_kernel<false><<<bx, 256, 0, st>>>(p);
    AVB_CUDA_OK(cudaGetLastError());
    return AVB_OK;
}

extern "C" int avb_uv_map_f32(const float *ubg_dev, void *out, int out_is_f32, int quantize, int n, int H, int W,
                              int64_t out_frame_stride, int64_t out_row_stride, const uint32_t *enc_dev,
                              int map_mode, const float *map_params_host, float mix_alpha,
                              void *workspace_dev, avb_stream_t stream) {
    AVB_REQUIRE(ubg_dev && out && workspace_dev, "null pointer");
    AVB_REQUIRE((reinterpret_cast<uintptr_t>(workspace_dev) & 15) == 0, "workspace_dev must be 16-byte aligned");
    AVB_REQUIRE(n > 0 && n <= 65535 && H > 0 && W > 0 && (long long)H * W < (1LL << 31), "bad frame geometry");
    AVB_REQUIRE(out_is_f32 || (enc_dev && out_row_stride >= 3LL * W), "uint8 output needs the encode table and a row stride >= 3*W");
    AVB_REQUIRE(map_mode >= 0 && map_mode <= MAP_MIXED, "unknown map_mode");
    AVB_REQUIRE(map_mode == MAP_OPPONENT || map_mode == MAP_FALSECOLOR || map_params_host, "this map_mode needs map_params_host");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    PlaneP pp{};
    pp.ubg = ubg_dev; pp.out = out; pp.out_f32 = out_is_f32; pp.quantize = quantize;
    UvParams &p = pp.uv;
    p.io = FrameIO{nullptr, out_is_f32 ? nullptr : static_cast<uint8_t *>(out), 0, 0, out_frame_stride, out_row_stride, n, H, W};
    p.enc = enc_dev;
    p.adapt = 0;
    p.eps = 1e-8f;
    p.mapper = map_mode;
    if (map_params_host) {
        for (int i = 0; i < 9; ++i) p.map_m[i] = map_params_host[i];
        for (int i = 0; i < 6; ++i) p.anchors[i] = map_params_host[9 + i];
    }
    p.mix_alpha = mix_alpha;
    const long long npx = (long long)H * W;
    uint8_t *ws = static_cast<uint8_t *>(workspace_dev);
    const size_t stats_bytes = align_up((size_t)n * sizeof(UvFrameStats), 256);
    const size_t hist_bytes = (size_t)n * UV_NH * UV_BINS * sizeof(uint32_t);
    const size_t planes_bytes = n_requests(map_mode) ? (size_t)n * UV_NH * (size_t)npx * sizeof(float) : 0;
    p.stats = reinterpret_cast<UvFrameStats *>(ws);
    p.hist = reinterpret_cast<uint32_t *>(ws + stats_bytes);
    p.planes = reinterpret_cast<float *>(ws + stats_bytes + hist_bytes);
    p.cand = reinterpret_cast<float *>(ws + stats_bytes + hist_bytes + planes_bytes);
    p.cap = npx;
    p.n_req = n_requests(map_mode);
    const double pcts[5][UV_NR] = {{95, 95, 0, 0}, {95, 95, 95, 0}, {0, 0, 0, 0}, {98, 0, 0, 0}, {95, 95, 95, 98}};
    const int hists[5][UV_NR] = {{0, 1, 0, 0}, {0, 1, 2, 0}, {0, 0, 0, 0}, {0, 0, 0, 0}, {0, 1, 2, 0}};
    for (int r = 0; r < p.n_req; ++r) {
        const PctIndex pi = numpy_percentile_index(pcts[map_mode][r], npx);    // float32 virtual index, as NumPy computes it
        p.req_hist[r] = hists[map_mode][r];
        p.k_lo[r] = pi.k_lo; p.k_hi[r] = pi.k_hi; p.gamma[r] = pi.gamma;
    }
    AVB_CUDA_OK(cudaMemsetAsync(ws, 0, stats_bytes + hist_bytes, st));
    switch (map_mode) {
        case MAP_OPPONENT: return launch_mapper_f32<MAP_OPPONENT>(pp, st);
        case MAP_FALSECOLOR: return launch_mapper_f32<MAP_FALSECOLOR>(pp, st);
        case MAP_MATRIX: return launch_mapper_f32<MAP_MATRIX>(pp, st);
        case MAP_PURPLE: return launch_mapper_f32<MAP_PURPLE>(pp, st);
        default: return launch_mapper_f32<MAP_MIXED>(pp, st);
    }
}
