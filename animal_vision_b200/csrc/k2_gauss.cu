// K2: fused  producer -> separable Gaussian (REFLECT_101) -> clip -> sRGB encode -> uint8.
//
// One CTA (384 threads) owns a vertical strip of 128 pixels and streams down a segment of rows in
// blocks of 8 input rows.  Per block:
//   produce   decode + 3x3 into a planar fp32 tile with an R-pixel x halo.  The packed uint8 rows of a
//             block (strip + halo columns, REFLECT_101 halo rows resolved per row) are staged by the
//             TMA engine: one cp.async.bulk per row into a double-buffered raw byte tile, completion
//             on an mbarrier, issued one block ahead -- no thread waits on a global load.  The LUT
//             kernel then decodes 4 pixels (12 bytes) per thread, the cat warp kernel gathers its
//             bilinear taps from the tile; unaligned frames and image-border strips go pixel by pixel;
//   H pass    8 outputs per thread from an (8+2R)-wide register window (LDS.128), taps from the
//             kernel-parameter constant bank;
//   V pass    accumulator ("scatter") form: every thread owns one (column, channel) and keeps the
//             2R partial sums of the output rows still in flight in registers -- one LDS and 2R+1
//             FMAs per input row, no window shifting;
//   encode -> packed uint8 staging -> 128-bit stores.
// The fp32 intermediate never leaves shared memory: HBM sees the uint8 frame once in and once out
// (6 B/px).
//
// Two-plane mode: every dichromat matrix of the reference (collapse_LMS_matrix, animal_utils.py:
// 88-119, and the cat's L/M merge) has rank 2 -- L and M are merged before the way back to RGB --
// so T = P(3x2) Q(2x3) and blur(T x) = P blur(Q x): only TWO planes are produced and blurred (a
// third fewer FMAs), the 3x2 expansion happens in the encode phase.  Full-rank matrices take the
// three-plane instantiation.
//
// Two kernels share the H pass, V pass and encode: gauss_stream_kernel produces with DogProducer (LUT
// decode + 3x3; animals/dog.py:35-48), cat_warp_kernel with the binocular wide-FOV gather + blend + pow
// decode + 3x3 (animals/cat_widevision_utils.py:46-99, animals/cat.py:95-101).
#include <algorithm>
#include <cmath>
#include <cstdlib>

#include <cuda_fp16.h>

#include "avb_common.cuh"

namespace avb {

constexpr int G_TW = 128;       // strip width in pixels
constexpr int G_RB = 8;         // rows per block
constexpr int G_THREADS_PER_PLANE = 128;  // H pass (plane, row, 8-px group); V pass (plane, column)
constexpr int G_MAX_TAPS = 33;
constexpr int G_ENC_SMEM = AVB_ENC_TABLE_MAX;  // uint32 words reserved for the encode table

constexpr int g_round_pitch(int v) { return (v % 8 == 4) ? v : (v + ((12 - v % 8) % 8)); }

template <int R>
struct GaussCfg {
    static constexpr int WIN = G_RB + 2 * R;                          // columns used by 8 H outputs
    static constexpr int NW4 = (WIN + 3) / 4;                         // float4 loads per horizontal window
    static constexpr int IN_W = G_TW + 2 * R;                         // produced columns per row
    static constexpr int GROUPS = (IN_W + 3) / 4;                     // 4-pixel decode groups per row
    static constexpr int SP_WIN = (G_TW - 8) + 4 * NW4;               // furthest column the H window reads
    static constexpr int SP_MIN = SP_WIN > 4 * GROUPS ? SP_WIN : 4 * GROUPS;
    static constexpr int S_PITCH = g_round_pitch(SP_MIN);             // % 8 == 4: odd multiple of 16 B, conflict-free LDS.128
    static constexpr int X_PITCH = G_TW + 4;
    static constexpr int S_PLANE = G_RB * S_PITCH;                    // floats per plane
    static constexpr int X_PLANE = G_RB * X_PITCH;
};

struct GaussCommon {
    FrameIO io;
    float P[6];            // two-plane mode: rgb[c] = P[2c] * plane0 + P[2c+1] * plane1 (rank-2 colour matrix)
    float taps[G_MAX_TAPS];
    const uint32_t *enc;   // encode table (device)
    uint32_t *flags;       // per-frame "some byte >= 2" (AVB_NORM_AUTO) or nullptr
    int seg_h;             // rows per segment (multiple of G_RB)
    int fixup;             // 1: second launch, only frames whose flag stayed 0 are (re)processed
    int radius;            // tensor-core variant: the radius is a run-time value there
};

// ------------------------------------------------------------------------------------ producers
struct DogProducer {
    static const char *name() { return "k2_gauss_dichromat"; }
    static const char *fixup_name() { return "k2_gauss_dichromat_fixup"; }
    struct Params {
        Mat3 M;
        const float *lut;  // 256-entry decode LUT (device)
    };
    static constexpr int SMEM_FLOATS = 256;
    static constexpr int RAW_PITCH = 528;  // bytes per row of the raw tile: 33 chunks of 16 B
    const float *lut_s;
    const uint8_t *src;
    int64_t rs;
    float m[9];
    uint32_t seen;

    __device__ __forceinline__ void init(const Params &pp, float *smem, const uint8_t *frame, int64_t row_stride,
                                         int /*H*/, int /*W*/, int /*frame_idx*/) {
        for (int i = threadIdx.x; i < 256; i += blockDim.x) smem[i] = __ldg(pp.lut + i);
        lut_s = smem;
        src = frame;
        rs = row_stride;
#pragma unroll
        for (int i = 0; i < 9; ++i) m[i] = pp.M.m[i];
        seen = 0;
    }
    __device__ __forceinline__ void px(uint32_t b0, uint32_t b1, uint32_t b2, float &o0, float &o1, float &o2) const {
        const float l0 = lut_s[b0], l1 = lut_s[b1], l2 = lut_s[b2];
        o0 = m[0] * l0 + m[1] * l1 + m[2] * l2;
        o1 = m[3] * l0 + m[4] * l1 + m[5] * l2;
        o2 = m[6] * l0 + m[7] * l1 + m[8] * l2;
    }
    // 12 packed bytes (4 pixels) -> planar float4 per channel
    __device__ __forceinline__ void decode4(uint32_t w0, uint32_t w1, uint32_t w2, float4 &c0, float4 &c1, float4 &c2) {
        seen |= w0 | w1 | w2;
        px(__byte_perm(w0, 0, 0x4440), __byte_perm(w0, 0, 0x4441), __byte_perm(w0, 0, 0x4442), c0.x, c1.x, c2.x);
        px(__byte_perm(w0, 0, 0x4443), __byte_perm(w1, 0, 0x4440), __byte_perm(w1, 0, 0x4441), c0.y, c1.y, c2.y);
        px(__byte_perm(w1, 0, 0x4442), __byte_perm(w1, 0, 0x4443), __byte_perm(w2, 0, 0x4440), c0.z, c1.z, c2.z);
        px(__byte_perm(w2, 0, 0x4441), __byte_perm(w2, 0, 0x4442), __byte_perm(w2, 0, 0x4443), c0.w, c1.w, c2.w);
    }
    struct Column { int x3; };
    __device__ __forceinline__ Column column(int x) const { return Column{3 * x}; }
    __device__ __forceinline__ void at(const Column &c, int y, float &o0, float &o1, float &o2) {
        const uint8_t *q = src + (int64_t)y * rs + c.x3;
        const uint32_t b0 = q[0], b1 = q[1], b2 = q[2];
        seen |= b0 | b1 | b2;
        px(b0, b1, b2, o0, o1, o2);
    }
};

// ------------------------------------------------------------------------------------ bulk-copy (TMA) helpers
__device__ __forceinline__ uint32_t gauss_smem(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void gauss_mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(gauss_smem(bar)), "r"(count));
}
__device__ __forceinline__ void gauss_bulk_load(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(gauss_smem(bar)), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(gauss_smem(dst)), "l"(src), "r"(bytes), "r"(gauss_smem(bar)) : "memory");
}
__device__ __forceinline__ void gauss_mbar_wait(uint64_t *bar, uint32_t parity) {
    const uint32_t a = gauss_smem(bar);
    uint32_t ok = 0;
    while (!ok)
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(ok) : "r"(a), "r"(parity) : "memory");
}

// ------------------------------------------------------------------------------------ phases shared by both kernels
// H pass: thread -> (plane ch, row h_r, 8-px group h_xg); 8 outputs from a WIN-wide register window
template <int R>
__device__ __forceinline__ void gauss_hpass(const GaussCommon &p, const float *S, float *X, int ch, int h_r, int h_xg) {
    using C = GaussCfg<R>;
    const float4 *w4 = reinterpret_cast<const float4 *>(&S[ch * C::S_PLANE + h_r * C::S_PITCH + h_xg * 8]);
    float v[4 * C::NW4];
#pragma unroll
    for (int q = 0; q < C::NW4; ++q) {
        const float4 t = w4[q];
        v[4 * q] = t.x; v[4 * q + 1] = t.y; v[4 * q + 2] = t.z; v[4 * q + 3] = t.w;
    }
    float acc[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] = 0.f;
#pragma unroll
    for (int k = 0; k <= 2 * R; ++k) {
        const float tk = p.taps[k];
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[j] = fmaf(tk, v[j + k], acc[j]);
    }
    float4 *d4 = reinterpret_cast<float4 *>(&X[ch * C::X_PLANE + h_r * C::X_PITCH + h_xg * 8]);
    d4[0] = make_float4(acc[0], acc[1], acc[2], acc[3]);
    d4[1] = make_float4(acc[4], acc[5], acc[6], acc[7]);
}

// V pass, one input row at a time: finish the oldest output row, advance the rest.  Thread -> (plane ch, column v_x).
// Input row i (0-based in the segment) completes output row y_start + i - 2R.
template <int R>
__device__ __forceinline__ void gauss_vpass(const GaussCommon &p, const float *X, float *Y, int ch, int v_x, float (&A)[2 * R]) {
    using C = GaussCfg<R>;
    const float *col = X + ch * C::X_PLANE + v_x;
    float *ycol = Y + ch * C::X_PLANE + v_x;
#pragma unroll
    for (int r = 0; r < G_RB; ++r) {
        const float h = col[r * C::X_PITCH];
        ycol[r * C::X_PITCH] = fmaf(p.taps[2 * R], h, A[0]);
#pragma unroll
        for (int m = 0; m < 2 * R - 1; ++m) A[m] = fmaf(p.taps[2 * R - 1 - m], h, A[m + 1]);
        A[2 * R - 1] = p.taps[0] * h;
    }
}

// expand (two-plane mode) + encode + store: a task is 4 consecutive pixels of one row (12 bytes = three 32-bit
// stores); input row i = 8*ib + r -> output row y_start + i - 2R
template <int R, int NCH, int THREADS>
__device__ __forceinline__ void gauss_encode_store(const GaussCommon &p, const EncTable &enc, const float *Y, uint8_t *dst_frame,
                                                   int ib, int y_start, int y_end, int x0, bool out4) {
    using C = GaussCfg<R>;
    const int W = p.io.W;
    const int oy0 = y_start + ib * G_RB - 2 * R;
    for (int t = threadIdx.x; t < G_RB * (G_TW / 4); t += THREADS) {
        const int r = t >> 5, g4 = t & 31;
        const int oy = oy0 + r;
        if (oy < y_start || oy >= y_end) continue;
        const int xo = x0 + 4 * g4;
        if (xo >= W) continue;
        const float4 a4 = *reinterpret_cast<const float4 *>(&Y[0 * C::X_PLANE + r * C::X_PITCH + 4 * g4]);
        const float4 b4 = *reinterpret_cast<const float4 *>(&Y[1 * C::X_PLANE + r * C::X_PITCH + 4 * g4]);
        float4 c4 = make_float4(0.f, 0.f, 0.f, 0.f);
        if (NCH == 3) c4 = *reinterpret_cast<const float4 *>(&Y[2 * C::X_PLANE + r * C::X_PITCH + 4 * g4]);
        const float av[4] = {a4.x, a4.y, a4.z, a4.w}, bv[4] = {b4.x, b4.y, b4.z, b4.w}, cv[4] = {c4.x, c4.y, c4.z, c4.w};
        uint32_t by[12];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            float r0, r1, r2;
            if (NCH == 2) {
                r0 = fmaf(p.P[1], bv[j], p.P[0] * av[j]);
                r1 = fmaf(p.P[3], bv[j], p.P[2] * av[j]);
                r2 = fmaf(p.P[5], bv[j], p.P[4] * av[j]);
            } else {
                r0 = av[j]; r1 = bv[j]; r2 = cv[j];
            }
            by[3 * j] = encode_u8(enc, r0);
            by[3 * j + 1] = encode_u8(enc, r1);
            by[3 * j + 2] = encode_u8(enc, r2);
        }
        uint8_t *o = dst_frame + (int64_t)oy * p.io.out_rs + (int64_t)xo * 3;
        if (out4 && xo + 3 < W) {
            uint32_t *o32 = reinterpret_cast<uint32_t *>(o);
#pragma unroll
            for (int q = 0; q < 3; ++q) o32[q] = by[4 * q] | (by[4 * q + 1] << 8) | (by[4 * q + 2] << 16) | (by[4 * q + 3] << 24);
        } else {
            const int nb = 3 * min(4, W - xo);
#pragma unroll
            for (int q = 0; q < 12; ++q)
                if (q < nb) o[q] = (uint8_t)by[q];
        }
    }
}

// ------------------------------------------------------------------------------------ LUT kernel
#ifndef G_MINB
#define G_MINB 2
#endif
#ifndef G_MINB3_R
#define G_MINB3_R 14
#endif
// two-plane CTAs (256 threads) fit three per SM up to radius 14 (72 registers with the TMA-staged tiles);
// three-plane CTAs (384 threads) keep the earlier split
template <int R, int NCH>
struct GaussOcc { static constexpr int MIN_BLOCKS = (R <= (NCH == 2 ? G_MINB3_R : 8)) ? 3 : G_MINB; };

template <int R, int NCH>
__global__ void __launch_bounds__(G_THREADS_PER_PLANE * NCH, GaussOcc<R, NCH>::MIN_BLOCKS)
gauss_stream_kernel(const __grid_constant__ GaussCommon p, const __grid_constant__ DogProducer::Params pp) {
    using C = GaussCfg<R>;
    constexpr int THREADS = G_THREADS_PER_PLANE * NCH;
    extern __shared__ __align__(16) uint8_t smem_raw[];
    float *S = reinterpret_cast<float *>(smem_raw);            // [NCH][RB][S_PITCH] produced rows (+x halo)
    float *X = S + NCH * C::S_PLANE;                           // [NCH][RB][X_PITCH] horizontally blurred rows
    float *Y = X + NCH * C::X_PLANE;                           // [NCH][RB][X_PITCH] fully blurred rows
    float *prod_smem = Y + NCH * C::X_PLANE;
    uint32_t *enc_s = reinterpret_cast<uint32_t *>(prod_smem + DogProducer::SMEM_FLOATS);
    uint8_t *rawt0 = reinterpret_cast<uint8_t *>(enc_s + G_ENC_SMEM);              // [2][RB][RAW_PITCH] packed input rows (TMA double buffer)
    constexpr int RAW_PITCH = DogProducer::RAW_PITCH;
    __shared__ __align__(8) uint64_t rbar[2];                                       // completion of the bulk copies of each buffer

    const int frame = blockIdx.z;
    if (p.fixup && p.flags[frame] != 0) return;

    const int tid = threadIdx.x, lane = tid & 31;
    const int H = p.io.H, W = p.io.W;
    const int x0 = blockIdx.x * G_TW;
    const int y_start = blockIdx.y * p.seg_h;
    const int y_end = min(H, y_start + p.seg_h);

    DogProducer prod;
    const uint8_t *src_frame = p.io.in + (int64_t)frame * p.io.in_fs;
    prod.init(pp, prod_smem, src_frame, p.io.in_rs, H, W, frame);
    copy_to_smem(enc_s, p.enc, min(G_ENC_SMEM, ENC_HEADER + (int)__ldg(p.enc + 2)));
    __syncthreads();
    const EncTable enc = enc_view(enc_s);

    uint8_t *dst_frame = p.io.out + (int64_t)frame * p.io.out_fs;
    const bool out4 = ((p.io.out_rs & 3) == 0) && ((p.io.out_fs & 3) == 0) && ((reinterpret_cast<uintptr_t>(p.io.out) & 3) == 0);

    // Raw tile: the packed bytes [a0, a0 + 16*n_chunks) of 8 input rows -- the strip plus its halo (and the
    // over-read of the last 4-pixel group) -- fetched with 16-byte loads one block ahead.
    const bool in16 = ((p.io.in_rs & 15) == 0) && ((p.io.in_fs & 15) == 0) && ((reinterpret_cast<uintptr_t>(p.io.in) & 15) == 0);
    const int a_byte = 3 * (x0 - R);                 // first byte of the produced span
    const int a0 = a_byte & ~15;
    const int n_chunks = (a_byte - a0 + 12 * C::GROUPS + 15) >> 4;
    const bool vec_in = x0 - R >= 0 && a0 + 16 * n_chunks <= 3 * W && in16 && 16 * n_chunks <= RAW_PITCH;

    const int n_in_rows = (y_end - y_start) + 2 * R;
    const int n_in_blocks = (n_in_rows + G_RB - 1) / G_RB;

    // task coordinates.  H pass: thread -> (plane, row, 8-px group); V pass: thread -> (plane, column)
    const int ch = tid >> 7;                         // 128 threads per plane
    const int h_r = tid & 7, h_xg = (tid & 127) >> 3;
    const int v_x = tid & 127;
    float A[2 * R];                                  // partial sums of the 2R output rows in flight
#pragma unroll
    for (int i = 0; i < 2 * R; ++i) A[i] = 0.f;

    // Raw-tile staging: thread r < G_RB issues the bulk copy of row r of a block (bytes [a0, a0 + 16 n_chunks)
    // of input row reflect101(yb + r)) and arrives on the buffer's mbarrier with the byte count.
    if (tid == 0) {
        gauss_mbar_init(&rbar[0], G_RB);
        gauss_mbar_init(&rbar[1], G_RB);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    auto raw_issue = [&](int yb_, int buf) {
        if (tid < G_RB) {
            const uint8_t *g = src_frame + (int64_t)reflect101(yb_ + tid, H) * p.io.in_rs + a0;
            gauss_bulk_load(rawt0 + buf * (G_RB * RAW_PITCH) + tid * RAW_PITCH, g, 16u * (uint32_t)n_chunks, &rbar[buf]);
        }
    };
    uint32_t rphase = 0;                             // bit b: parity the next wait on buffer b expects
    if (vec_in) raw_issue(y_start - R, 0);

    for (int ib = 0; ib < n_in_blocks; ++ib) {
        const int yb = y_start - R + ib * G_RB;      // first input row of this block
        // ---- produce RB rows x IN_W columns of linear-light values
        if (vec_in) {
            // the packed rows of this block were requested one block ahead: wait for the copies, then put
            // the next block's copies in flight (its buffer was last read two barriers ago)
            const int buf = ib & 1;
            const uint8_t *rawt = rawt0 + buf * (G_RB * RAW_PITCH);
            gauss_mbar_wait(&rbar[buf], (rphase >> buf) & 1u);
            rphase ^= 1u << buf;
            if (ib + 1 < n_in_blocks) raw_issue(yb + G_RB, buf ^ 1);
            // a task is a group of 4 pixels; the tasks beyond the first THREADS are split into single
            // pixels (second round: one pixel per thread instead of four)
            constexpr int NTG = G_RB * C::GROUPS, REMG_ALL = NTG > THREADS ? NTG - THREADS : 0;
            // (measured: splitting pays while the remainder is small; with 56 left-over groups -- 29 taps --
            // the byte-granular second round costs as much as it saves)
            constexpr int REMG = REMG_ALL <= 32 ? REMG_ALL : 0;
            const int sh = (a_byte - a0) & 3, w_off = (a_byte - a0) >> 2;
            if (REMG > 0 && tid < 4 * REMG) {
                const int idx = NTG - REMG + (tid >> 2), j = tid & 3;
                const int r = idx / C::GROUPS, g = idx - r * C::GROUPS;
                const uint8_t *q = rawt + r * RAW_PITCH + (a_byte - a0) + 3 * (4 * g + j);
                const uint32_t b0 = q[0], b1 = q[1], b2 = q[2];
                prod.seen |= b0 | b1 | b2;
                float o0, o1, o2;
                prod.px(b0, b1, b2, o0, o1, o2);
                S[0 * C::S_PLANE + r * C::S_PITCH + 4 * g + j] = o0;
                S[1 * C::S_PLANE + r * C::S_PITCH + 4 * g + j] = o1;
                if (NCH == 3) S[2 * C::S_PLANE + r * C::S_PITCH + 4 * g + j] = o2;
            }
            for (int idx = tid; idx < NTG - REMG; idx += THREADS) {
                const int r = idx / C::GROUPS, g = idx - r * C::GROUPS;
                const uint32_t *q = reinterpret_cast<const uint32_t *>(rawt + r * RAW_PITCH) + w_off + 3 * g;
                uint32_t w0 = q[0], w1 = q[1], w2 = q[2];
                if (sh) {
                    const uint32_t w3 = q[3];
                    w0 = __funnelshift_r(w0, w1, 8 * sh);
                    w1 = __funnelshift_r(w1, w2, 8 * sh);
                    w2 = __funnelshift_r(w2, w3, 8 * sh);
                }
                float4 c0, c1, c2;
                prod.decode4(w0, w1, w2, c0, c1, c2);
                *reinterpret_cast<float4 *>(&S[0 * C::S_PLANE + r * C::S_PITCH + 4 * g]) = c0;
                *reinterpret_cast<float4 *>(&S[1 * C::S_PLANE + r * C::S_PITCH + 4 * g]) = c1;
                if (NCH == 3) *reinterpret_cast<float4 *>(&S[2 * C::S_PLANE + r * C::S_PITCH + 4 * g]) = c2;
            }
        } else {
            // pixel-by-pixel producer (image borders, unaligned frames): a task is one column x 4 rows
            for (int idx = tid; idx < 2 * C::IN_W; idx += THREADS) {
                const int half = idx / C::IN_W, i = idx - half * C::IN_W;
                const DogProducer::Column col = prod.column(reflect101(x0 - R + i, W));
#pragma unroll
                for (int rr = 0; rr < G_RB / 2; ++rr) {
                    const int r = half * (G_RB / 2) + rr;
                    float o0, o1, o2;
                    prod.at(col, reflect101(yb + r, H), o0, o1, o2);
                    S[0 * C::S_PLANE + r * C::S_PITCH + i] = o0;
                    S[1 * C::S_PLANE + r * C::S_PITCH + i] = o1;
                    if (NCH == 3) S[2 * C::S_PLANE + r * C::S_PITCH + i] = o2;
                }
            }
        }
        __syncthreads();
        gauss_hpass<R>(p, S, X, ch, h_r, h_xg);
        __syncthreads();
        gauss_vpass<R>(p, X, Y, ch, v_x, A);
        __syncthreads();
        gauss_encode_store<R, NCH, THREADS>(p, enc, Y, dst_frame, ib, y_start, y_end, x0, out4);
        // hazards: the next produce writes rawt / S (H pass done); X is rewritten after the next
        // produce barrier (V pass done); Y is rewritten after the next H-pass barrier (encode done).
    }

    if (p.flags != nullptr && !p.fixup) {
        // vector path ORs whole 32-bit words (4 packed bytes), the scalar path single bytes
        if (__any_sync(0xffffffffu, (prod.seen & 0xfefefefeu) != 0) && lane == 0) p.flags[frame] = 1u;
    }
}

// ------------------------------------------------------------------------------------ tensor-core variant
// The separable Gaussian of the two-plane LUT path as two banded-Toeplitz matrix products on the tensor cores
// (mma.sync m16n8k16, f16 operands, f32 accumulate): per output pixel and plane the CUDA cores used to issue
// 2 x (2R+1) FMAs (116 of Dog's 261 instructions per pixel); here a warp instruction retires 2 048 MACs.
// Register-fragment MMAs rather than tcgen05: the operator is BANDED, and a 16-wide output tile needs only
// K = 16 + 2R (padded to 32/48) inputs per output, where a 128-row UMMA tile would multiply 128 + 2R -- the
// tensor pipe would become the bound of an otherwise CUDA-core kernel (measured mma.sync rate on B200:
// 555 TFLOP/s, tools/micro/hmma_rate.cu; this kernel needs 0.13 TFLOP per 20 4K frames at 29 taps).
//
//   produce   as above (TMA-staged packed rows, LUT decode, 2x3 matrix) into a PLANAR F16 tile S[plane]
//             [16 rows][x halo]
//   H pass    D[16 rows x 8 cols] += S[16 rows x 16s..16s+15] * T_s,  T_s[k][n] = w[16s + k - n]: the Toeplitz
//             fragments are pixel independent and live in registers for the whole kernel (6 words)
//   ring      the H results (f16 again) of the last (D+1) blocks of 16 rows, D = ceil(2R/16)
//   V pass    D[16 out rows x 8 cols] += T'_s[16 x 16] * ring[block ob+s][16 rows x 8 cols] (ldmatrix.trans)
//   encode    expand the two planes, table encode, packed bytes staged in shared memory, 128-bit stores.
// Taps are rounded to f16 on the host with the rounding error diffused so that they still sum to 1 (flat
// regions stay exact); the accumulation is f32.
constexpr int M_RB = 16;            // rows per block (the M of the H pass, the N tile rows of the V pass)
constexpr int M_THREADS = 256;      // 8 warps: warp w owns output column tiles 2w, 2w+1 of both planes
constexpr int M_HP = 136;           // ring pitch in halves: 272 B = 17 x 16 B (ldmatrix rows hit distinct banks)
constexpr int M_STAGE_PITCH = 3 * G_TW + 16;   // 400 B = 100 words: the 8 fragment rows of a warp land in distinct banks
constexpr int M_RAW_PITCH = 512;
constexpr int M_LUT_COPIES = 4;     // decode LUT replicated: lane l reads copy l & 3 (random byte values spread over 4x the banks)

__device__ __forceinline__ void ldsm_x4(uint32_t (&r)[4], uint32_t addr) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void ldsm_x2(uint32_t (&r)[2], uint32_t addr) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x2.shared.b16 {%0,%1}, [%2];" : "=r"(r[0]), "=r"(r[1]) : "r"(addr));
}
__device__ __forceinline__ void ldsm_x4_trans(uint32_t (&r)[4], uint32_t addr) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void mma16816(float (&c)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3]) : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}
__device__ __forceinline__ uint32_t pack_h2(float a, float b) {
    const __half2 h = __floats2half2_rn(a, b);
    return *reinterpret_cast<const uint32_t *>(&h);
}

template <int KSH>
struct MmaCfg {
    static constexpr int SP = 120 + 16 * KSH;     // S pitch in halves: 304 / 336 B = 19 / 21 x 16 B
};

struct MmaGeom {
    int radius, r4;        // blur radius; left halo of the produced tile = radius rounded up to 4 px (word-aligned packed rows)
    int groups;            // 4-pixel decode groups per row: ceil((128 + r4 + radius) / 4)
    uint32_t div_groups;   // ceil(2^16 / groups): idx / groups == (idx * div_groups) >> 16 for idx < 16 * groups
};

#ifndef M_MINB_SINGLE
#define M_MINB_SINGLE 3     // 71 registers and ~72 KB of shared memory per CTA, three CTAs per SM
#endif
template <int KSH, int D>
__global__ void __launch_bounds__(M_THREADS, M_MINB_SINGLE)
gauss_mma_kernel(const __grid_constant__ GaussCommon p, const __grid_constant__ DogProducer::Params pp, const __grid_constant__ MmaGeom geo) {
    constexpr int SP = MmaCfg<KSH>::SP;
    constexpr int KSV = D + 1;                    // k-steps of the V pass = ring depth in blocks
    constexpr int S_PLANE = M_RB * SP;            // halves per plane
    constexpr int H_PLANE = KSV * M_RB * M_HP;
    extern __shared__ __align__(128) uint8_t smem_raw[];
    __half *S = reinterpret_cast<__half *>(smem_raw);                     // [2][16][SP]
    __half *HR = S + 2 * S_PLANE;                                          // [2][KSV*16][M_HP]
    uint8_t *stage = reinterpret_cast<uint8_t *>(HR + 2 * H_PLANE);        // [16][400] encoded bytes of an output block
    float *lut4 = reinterpret_cast<float *>(stage + M_RB * M_STAGE_PITCH); // [256][M_LUT_COPIES]
    uint32_t *enc_s = reinterpret_cast<uint32_t *>(lut4 + 256 * M_LUT_COPIES);
    uint8_t *rawt0 = reinterpret_cast<uint8_t *>(enc_s + G_ENC_SMEM);      // [2][16][M_RAW_PITCH] packed input rows (TMA double buffer)
    __shared__ __align__(8) uint64_t rbar[2];

    const int frame = blockIdx.z;
    if (p.fixup && p.flags[frame] != 0) return;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int g = lane >> 2, t = lane & 3;
    const int H = p.io.H, W = p.io.W, R = geo.radius, R4 = geo.r4;
    const int x0 = blockIdx.x * G_TW;
    const int y_start = blockIdx.y * p.seg_h;
    const int y_end = min(H, y_start + p.seg_h);
    const int GROUPS = geo.groups, IN_W = 4 * GROUPS;

    const uint8_t *src_frame = p.io.in + (int64_t)frame * p.io.in_fs;
    for (int i = tid; i < 256 * M_LUT_COPIES; i += M_THREADS) lut4[i] = __ldg(pp.lut + (i / M_LUT_COPIES));
    copy_to_smem(enc_s, p.enc, min(G_ENC_SMEM, ENC_HEADER + (int)__ldg(p.enc + 2)));
    // the pad columns of S only ever meet zero Toeplitz entries, but they must hold finite numbers
    for (int i = tid; i < S_PLANE; i += M_THREADS) reinterpret_cast<uint32_t *>(S)[i] = 0u;
    if (tid == 0) {
        gauss_mbar_init(&rbar[0], M_RB);
        gauss_mbar_init(&rbar[1], M_RB);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    const EncTable enc = enc_view(enc_s);
    const float *lut_l = lut4 + (lane & (M_LUT_COPIES - 1));
    float qm[6];
#pragma unroll
    for (int i = 0; i < 6; ++i) qm[i] = pp.M.m[i];
    uint32_t seen = 0;
    auto px2 = [&](uint32_t b0, uint32_t b1, uint32_t b2, float &o0, float &o1) {
        const float l0 = lut_l[M_LUT_COPIES * b0], l1 = lut_l[M_LUT_COPIES * b1], l2 = lut_l[M_LUT_COPIES * b2];
        o0 = qm[0] * l0 + qm[1] * l1 + qm[2] * l2;         // same expression as DogProducer::px
        o1 = qm[3] * l0 + qm[4] * l1 + qm[5] * l2;
    };

    // Toeplitz fragments, f16x2, zero outside the taps.  H pass (S column i = image column x0 - R4 + i, so the taps
    // start R4 - R columns into the window): k-step s: b0 = th[2s], b1 = th[2s+1], th[j] = (w[8j + 2t - g - off], next).
    // V pass k-step s: a0 = a3 = tv[2s], a1 = tv[2s-1], a2 = tv[2s+1], tv[j] = (w[8j + 2t - g], next).
    uint32_t th[2 * KSH], tv[2 * KSV];
    {
        const int off = R4 - R;
        auto wt = [&](int i) { return (i >= 0 && i <= 2 * R) ? p.taps[i] : 0.f; };
#pragma unroll
        for (int j = 0; j < 2 * KSH; ++j) th[j] = pack_h2(wt(8 * j + 2 * t - g - off), wt(8 * j + 2 * t - g - off + 1));
#pragma unroll
        for (int j = 0; j < 2 * KSV; ++j) tv[j] = pack_h2(wt(8 * j + 2 * t - g), wt(8 * j + 2 * t - g + 1));
    }

    uint8_t *dst_frame = p.io.out + (int64_t)frame * p.io.out_fs;
    const bool vec_ok = (x0 + G_TW <= W) && ((p.io.out_rs & 15) == 0) && ((p.io.out_fs & 15) == 0) &&
                        ((reinterpret_cast<uintptr_t>(p.io.out) & 15) == 0);
    const bool in16 = ((p.io.in_rs & 15) == 0) && ((p.io.in_fs & 15) == 0) && ((reinterpret_cast<uintptr_t>(p.io.in) & 15) == 0);
    // Interior strips: the produced span [x0 - R4, x0 - R4 + IN_W) lies inside the row; its packed bytes start word aligned.
    // Border strips: the in-image part of the span is staged, REFLECT_101 columns are resolved against the staged bytes.
    const int c_lo = max(0, x0 - R4), c_hi = min(W, x0 - R4 + IN_W);
    const int a_byte = 3 * (x0 - R4);
    const int a0 = (3 * c_lo) & ~15;
    const int n_chunks = (3 * c_hi - a0 + 15) >> 4;
    const bool interior = x0 - R4 >= 0 && x0 - R4 + IN_W <= W;
    // every reflected column of a border strip must fall inside the staged span
    const bool refl_ok = reflect101(x0 - R4, W) < c_hi && reflect101(x0 - R4 + IN_W - 1, W) >= c_lo && W > IN_W;
    const bool staged = in16 && 16 * n_chunks <= M_RAW_PITCH && a0 + 16 * n_chunks <= 3 * W && ((a_byte & 3) == 0) && (interior || refl_ok);

    const int n_out_blocks = (y_end - y_start + M_RB - 1) / M_RB;
    const int n_blocks = n_out_blocks + D;

    auto raw_issue = [&](int ib_, int buf) {
        if (tid < M_RB) {
            const uint8_t *gsrc = src_frame + (int64_t)reflect101(y_start - R + ib_ * M_RB + tid, H) * p.io.in_rs + a0;
            gauss_bulk_load(rawt0 + buf * (M_RB * M_RAW_PITCH) + tid * M_RAW_PITCH, gsrc, 16u * (uint32_t)n_chunks, &rbar[buf]);
        }
    };
    uint32_t rphase = 0;
    if (staged) raw_issue(0, 0);

    const uint32_t S_sh = gauss_smem(S), HR_sh = gauss_smem(HR);
    // ldmatrix lane roles: matrix mi = lane >> 3, row (lane & 7) + 8 (mi & 1), second half of the pair mi >> 1
    const int l_row = (lane & 7) + 8 * ((lane >> 3) & 1), l_hi = lane >> 4;

    auto store_px = [&](int r, int i, float o0, float o1) {
        S[r * SP + i] = __float2half_rn(o0);
        S[S_PLANE + r * SP + i] = __float2half_rn(o1);
    };

    // ---- produce block ib: 16 rows x IN_W columns of the two planes as f16
    auto produce = [&](int ib) {
        const int yb = y_start - R + ib * M_RB;
        if (staged) {
            const int buf = ib & 1;
            const uint8_t *rawt = rawt0 + buf * (M_RB * M_RAW_PITCH);
            gauss_mbar_wait(&rbar[buf], (rphase >> buf) & 1u);
            rphase ^= 1u << buf;
            if (ib + 1 < n_blocks) raw_issue(ib + 1, buf ^ 1);
            if (interior) {
                const int w_off = (a_byte - a0) >> 2;
                for (int idx = tid; idx < M_RB * GROUPS; idx += M_THREADS) {
                    const int r = (int)(((uint32_t)idx * geo.div_groups) >> 16), gq = idx - r * GROUPS;
                    const uint32_t *q = reinterpret_cast<const uint32_t *>(rawt + r * M_RAW_PITCH) + w_off + 3 * gq;
                    const uint32_t w0 = q[0], w1 = q[1], w2 = q[2];
                    seen |= w0 | w1 | w2;
                    float a[4], b[4];
                    px2(__byte_perm(w0, 0, 0x4440), __byte_perm(w0, 0, 0x4441), __byte_perm(w0, 0, 0x4442), a[0], b[0]);
                    px2(__byte_perm(w0, 0, 0x4443), __byte_perm(w1, 0, 0x4440), __byte_perm(w1, 0, 0x4441), a[1], b[1]);
                    px2(__byte_perm(w1, 0, 0x4442), __byte_perm(w1, 0, 0x4443), __byte_perm(w2, 0, 0x4440), a[2], b[2]);
                    px2(__byte_perm(w2, 0, 0x4441), __byte_perm(w2, 0, 0x4442), __byte_perm(w2, 0, 0x4443), a[3], b[3]);
                    __half *d0 = S + r * SP + 4 * gq, *d1 = d0 + S_PLANE;
                    *reinterpret_cast<uint2 *>(d0) = make_uint2(pack_h2(a[0], a[1]), pack_h2(a[2], a[3]));
                    *reinterpret_cast<uint2 *>(d1) = make_uint2(pack_h2(b[0], b[1]), pack_h2(b[2], b[3]));
                }
            } else {
                for (int idx = tid; idx < M_RB * IN_W; idx += M_THREADS) {
                    const int r = (int)(((uint32_t)(idx >> 2) * geo.div_groups) >> 16), i = idx - r * IN_W;
                    const uint8_t *q = rawt + r * M_RAW_PITCH + 3 * reflect101(x0 - R4 + i, W) - a0;
                    const uint32_t b0 = q[0], b1 = q[1], b2 = q[2];
                    seen |= b0 | b1 | b2;
                    float o0, o1;
                    px2(b0, b1, b2, o0, o1);
                    store_px(r, i, o0, o1);
                }
            }
        } else {
            // unaligned frames, frames narrower than the tile: pixel by pixel from global memory
            for (int idx = tid; idx < M_RB * IN_W; idx += M_THREADS) {
                const int r = (int)(((uint32_t)(idx >> 2) * geo.div_groups) >> 16), i = idx - r * IN_W;
                const uint8_t *q = src_frame + (int64_t)reflect101(yb + r, H) * p.io.in_rs + 3 * reflect101(x0 - R4 + i, W);
                const uint32_t b0 = q[0], b1 = q[1], b2 = q[2];
                seen |= b0 | b1 | b2;
                float o0, o1;
                px2(b0, b1, b2, o0, o1);
                store_px(r, i, o0, o1);
            }
        }
    };

    // ---- H pass of block ib into ring slot ib % KSV
    auto hpass = [&](int ib) {
        const int slot = ib % KSV;
#pragma unroll
        for (int pl = 0; pl < 2; ++pl) {
            float acc[2][4];
#pragma unroll
            for (int e = 0; e < 2; ++e)
#pragma unroll
                for (int c = 0; c < 4; ++c) acc[e][c] = 0.f;
            // half-fragments (16 rows x 8 columns) at columns 16 warp + 8 h, h = 0 .. 2 KSH
            uint32_t hf[2 * KSH + 1][2];
            const uint32_t base = S_sh + 2u * (uint32_t)(pl * S_PLANE + l_row * SP + 16 * warp);
#pragma unroll
            for (int q = 0; q < KSH; ++q) {
                uint32_t r4[4];
                ldsm_x4(r4, base + 2u * (uint32_t)(16 * q + 8 * l_hi));
                hf[2 * q][0] = r4[0]; hf[2 * q][1] = r4[1]; hf[2 * q + 1][0] = r4[2]; hf[2 * q + 1][1] = r4[3];
            }
            {
                uint32_t r2[2];
                ldsm_x2(r2, base + 2u * (uint32_t)(16 * KSH));
                hf[2 * KSH][0] = r2[0]; hf[2 * KSH][1] = r2[1];
            }
#pragma unroll
            for (int e = 0; e < 2; ++e)
#pragma unroll
                for (int s = 0; s < KSH; ++s)
                    mma16816(acc[e], hf[2 * s + e][0], hf[2 * s + e][1], hf[2 * s + e + 1][0], hf[2 * s + e + 1][1], th[2 * s], th[2 * s + 1]);
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                __half *d = HR + pl * H_PLANE + (slot * M_RB + g) * M_HP + 8 * (2 * warp + e) + 2 * t;
                *reinterpret_cast<uint32_t *>(d) = pack_h2(acc[e][0], acc[e][1]);
                *reinterpret_cast<uint32_t *>(d + 8 * M_HP) = pack_h2(acc[e][2], acc[e][3]);
            }
        }
    };

    // ---- V pass of output block ob (window = ring blocks ob .. ob + D), expand the two planes, encode, stage
    auto vencode = [&](int ob) {
        float out[2][2][4];                        // [plane][column tile][fragment]
#pragma unroll
        for (int pl = 0; pl < 2; ++pl) {
#pragma unroll
            for (int e = 0; e < 2; ++e)
#pragma unroll
                for (int c = 0; c < 4; ++c) out[pl][e][c] = 0.f;
#pragma unroll
            for (int s = 0; s < KSV; ++s) {
                const int slot = (ob + s) % KSV;
                uint32_t b4[4];
                ldsm_x4_trans(b4, HR_sh + 2u * (uint32_t)(pl * H_PLANE + (slot * M_RB + l_row) * M_HP + 8 * (2 * warp + l_hi)));
                const uint32_t a1 = s > 0 ? tv[2 * s - 1] : 0u;
                mma16816(out[pl][0], tv[2 * s], a1, tv[2 * s + 1], tv[2 * s], b4[0], b4[1]);
                mma16816(out[pl][1], tv[2 * s], a1, tv[2 * s + 1], tv[2 * s], b4[2], b4[3]);
            }
        }
        // fragment: (row g / g+8, columns 2t, 2t+1) of column tiles 2 warp, 2 warp + 1
#pragma unroll
        for (int e = 0; e < 2; ++e)
#pragma unroll
            for (int hh = 0; hh < 2; ++hh) {
                uint32_t by[6];
#pragma unroll
                for (int j = 0; j < 2; ++j) {
                    const float av = out[0][e][2 * hh + j], bv = out[1][e][2 * hh + j];
                    by[3 * j] = encode_u8(enc, fmaf(p.P[1], bv, p.P[0] * av));
                    by[3 * j + 1] = encode_u8(enc, fmaf(p.P[3], bv, p.P[2] * av));
                    by[3 * j + 2] = encode_u8(enc, fmaf(p.P[5], bv, p.P[4] * av));
                }
                uint16_t *o = reinterpret_cast<uint16_t *>(stage + (g + 8 * hh) * M_STAGE_PITCH + 3 * (8 * (2 * warp + e) + 2 * t));
                o[0] = (uint16_t)(by[0] | (by[1] << 8));
                o[1] = (uint16_t)(by[2] | (by[3] << 8));
                o[2] = (uint16_t)(by[4] | (by[5] << 8));
            }
    };

    // ---- staged rows of output block ob -> global
    auto copy_out = [&](int ob) {
        const int oy0 = y_start + ob * M_RB;
        if (vec_ok) {
            constexpr int CH = 3 * G_TW / 16;          // 24 chunks of 16 B per row
            for (int idx = tid; idx < M_RB * CH; idx += M_THREADS) {
                const int r = idx / CH, c = idx - r * CH;
                if (oy0 + r < y_end)
                    *reinterpret_cast<uint4 *>(dst_frame + (int64_t)(oy0 + r) * p.io.out_rs + (int64_t)x0 * 3 + 16 * c) =
                        *reinterpret_cast<const uint4 *>(stage + r * M_STAGE_PITCH + 16 * c);
            }
        } else {
            const int nbytes = 3 * min(G_TW, W - x0);
            for (int idx = tid; idx < M_RB * 3 * G_TW; idx += M_THREADS) {
                const int r = idx / (3 * G_TW), b = idx - r * (3 * G_TW);
                if (oy0 + r < y_end && b < nbytes) dst_frame[(int64_t)(oy0 + r) * p.io.out_rs + (int64_t)x0 * 3 + b] = stage[r * M_STAGE_PITCH + b];
            }
        }
    };

    // Two barriers per 16-row block, each interval mixing two kinds of work:
    //   B(ib): H pass of block ib (tensor + LDSM)      + copy-out of output block ib-1-D (LDS.128 / STG.128)
    //   A(ib): produce block ib+1 (LDS, LUT, FMA, F2FP) + V pass / encode of output block ib-D (tensor, ALU)
    // S is written in A and read in B; ring slot ib % KSV is written in B(ib) and last read in A(ib+D); the byte
    // stage is written in A and read in the following B.
    produce(0);
    __syncthreads();
    for (int ib = 0; ib < n_blocks; ++ib) {
        hpass(ib);
        if (ib - 1 - D >= 0) copy_out(ib - 1 - D);
        __syncthreads();
        if (ib + 1 < n_blocks) produce(ib + 1);
        if (ib >= D) vencode(ib - D);
        __syncthreads();
    }
    copy_out(n_blocks - 1 - D);

    if (p.flags != nullptr && !p.fixup) {
        if (__any_sync(0xffffffffu, (seen & 0xfefefefeu) != 0) && lane == 0) p.flags[frame] = 1u;
    }
}

template <int R, int NCH>
static int launch_gauss(const GaussCommon &gc, const DogProducer::Params &pp, cudaStream_t st) {
    using C = GaussCfg<R>;
    const size_t smem = (size_t)(NCH * C::S_PLANE + 2 * NCH * C::X_PLANE + DogProducer::SMEM_FLOATS + G_ENC_SMEM) * 4 + 2 * (size_t)G_RB * DogProducer::RAW_PITCH;
    auto kern = gauss_stream_kernel<R, NCH>;
    AVB_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    dim3 grid((gc.io.W + G_TW - 1) / G_TW, (gc.io.H + gc.seg_h - 1) / gc.seg_h, gc.io.n);
    AVB_TIMED(gc.fixup ? DogProducer::fixup_name() : DogProducer::name(), st);
    kern<<<grid, G_THREADS_PER_PLANE * NCH, smem, st>>>(gc, pp);
    AVB_CUDA_OK(cudaGetLastError());
    return AVB_OK;
}

// Rows per segment.  Every CTA of a launch does the same amount of work, so the launch runs in waves of
// (SMs x resident CTAs per SM): the segment count is chosen to maximise
//     (fill of the last wave) x (useful rows / produced rows),
// i.e. it trades the 2R halo rows re-produced per segment against a nearly empty last wave (1 800 CTAs on
// 296 slots run seven waves, the seventh 8 % full).
static int pick_seg_h(int n, int H, int W, int radius, int ctas_per_sm) {
    const long strips = (long)((W + G_TW - 1) / G_TW) * n;
    const long slots = (long)sm_count() * ctas_per_sm;
    const int min_h = std::max(G_RB, 8 * radius);               // halo rows re-produced per segment <= 25 %
    const int max_segs = std::max(1, (H + min_h - 1) / min_h);
    int best = 1;
    double best_score = -1.0;
    for (int segs = 1; segs <= max_segs && segs <= 64; ++segs) {
        int seg_h = (H + segs - 1) / segs;
        seg_h = (seg_h + G_RB - 1) / G_RB * G_RB;
        const long real_segs = (H + seg_h - 1) / seg_h;
        const long ctas = strips * real_segs;
        const long waves = (ctas + slots - 1) / slots;
        const double fill = (double)ctas / (double)(waves * slots);
        const double useful = (double)seg_h / (double)(seg_h + 2 * radius);
        // a launch of less than ~2 waves cannot hide its ramp-up: prefer more, smaller CTAs there
        const double score = fill * useful * (waves >= 2 ? 1.0 : 0.85);
        if (score > best_score + 1e-9) { best_score = score; best = segs; }
    }
    int seg_h = (H + best - 1) / best;
    return (seg_h + G_RB - 1) / G_RB * G_RB;
}

// T (3x3, applied as out = T lin) = P (3x2) Q (2x3) if it has rank <= 2: Q = the two most independent
// rows of T (exact copies), P = the coefficients of every row in that basis (least squares, double).
// Returns false for a full-rank matrix (residual above float32 rounding of T itself).
static bool rank2_factor(const float *T, float *Q /*6*/, float *P /*6*/) {
    double r[3][3];
    for (int i = 0; i < 9; ++i) r[i / 3][i % 3] = T[i];
    int bi = 0, bj = 1;
    double best = -1.0;
    for (int i = 0; i < 3; ++i)
        for (int j = i + 1; j < 3; ++j) {
            const double cx = r[i][1] * r[j][2] - r[i][2] * r[j][1], cy = r[i][2] * r[j][0] - r[i][0] * r[j][2],
                         cz = r[i][0] * r[j][1] - r[i][1] * r[j][0];
            const double n2 = cx * cx + cy * cy + cz * cz;
            if (n2 > best) { best = n2; bi = i; bj = j; }
        }
    const double aa = r[bi][0] * r[bi][0] + r[bi][1] * r[bi][1] + r[bi][2] * r[bi][2];
    const double bb = r[bj][0] * r[bj][0] + r[bj][1] * r[bj][1] + r[bj][2] * r[bj][2];
    const double ab = r[bi][0] * r[bj][0] + r[bi][1] * r[bj][1] + r[bi][2] * r[bj][2];
    const double det = aa * bb - ab * ab;
    double scale = 0.0;
    for (int i = 0; i < 9; ++i) scale = std::max(scale, std::fabs((double)T[i]));
    if (!(det > 1e-12 * scale * scale * scale * scale)) return false;      // rank <= 1: not worth a special case
    double resid = 0.0;
    for (int k = 0; k < 3; ++k) {
        const double ka = r[k][0] * r[bi][0] + r[k][1] * r[bi][1] + r[k][2] * r[bi][2];
        const double kb = r[k][0] * r[bj][0] + r[k][1] * r[bj][1] + r[k][2] * r[bj][2];
        double c0 = (ka * bb - kb * ab) / det, c1 = (kb * aa - ka * ab) / det;
        if (k == bi) { c0 = 1.0; c1 = 0.0; }
        if (k == bj) { c0 = 0.0; c1 = 1.0; }
        P[2 * k] = (float)c0; P[2 * k + 1] = (float)c1;
        for (int c = 0; c < 3; ++c) resid = std::max(resid, std::fabs(r[k][c] - ((double)P[2 * k] * r[bi][c] + (double)P[2 * k + 1] * r[bj][c])));
    }
    for (int c = 0; c < 3; ++c) { Q[c] = T[3 * bi + c]; Q[3 + c] = T[3 * bj + c]; }
    return resid <= 4e-7 * scale;       // a few float32 ulps of the largest entry: T itself was rounded to float32
}

// ---- tensor-core variant: host side
// Taps -> f16 with the rounding error diffused: every tap is rounded to f16, then symmetric pairs are nudged by whole
// f16 steps, largest step first, until the taps sum to 1 within the finest step.  A flat region then blurs to
// itself exactly (f32 accumulation), as it does in the reference.
static double f16_step(double v) {
    v = std::fabs(v);
    if (v < 6.103515625e-05) return 5.960464477539063e-08;          // subnormal spacing 2^-24
    int e;
    std::frexp(v, &e);                                               // v = m 2^e, m in [0.5, 1)
    return std::ldexp(1.0, e - 11);
}
static void quantize_taps_f16(float *taps, int ksize) {
    const int c = ksize / 2;
    double q[G_MAX_TAPS];
    for (int i = 0; i < ksize; ++i) q[i] = (double)__half2float(__float2half_rn(taps[i]));
    double sum = 0.0;
    for (int i = 0; i < ksize; ++i) sum += q[i];
    for (int k = 0; k <= c; ++k) {                                   // centre (largest step) outwards
        const double step = f16_step(q[c + k]) * (k ? 2.0 : 1.0);
        const double m = std::nearbyint((1.0 - sum) / step);
        if (m == 0.0) continue;
        const double d = m * f16_step(q[c + k]);
        q[c + k] += d;
        if (k) q[c - k] += d;
        sum += m * step;
    }
    for (int i = 0; i < ksize; ++i) taps[i] = (float)q[i];
}

// A rank-2 matrix with radius 5..16 takes the tensor-core kernel.  Its single f16 operands cost ~0.05 LSB of systematic
// rounding: <= 1 LSB, with 0.3-1.4 % of the bytes differing (a flat region may flip by 1 LSB as a whole).  Measured, 20 4K
// frames, ms, against hi+lo f16 operands (Dog, Raccoon) or the CUDA-core kernel (the others): Dog (29 taps) 1.13 -> 0.85,
// Raccoon (17) 0.99 -> 0.77, Bear / Elephant (15) 1.03 -> 0.77, Wolf (13) / Fox / Lion (11) 0.91 -> 0.77.
// Squirrel (7 taps) would gain too (0.82 -> 0.75) but stays on the exact CUDA-core kernel: its narrow blur leaves the plateaus
// of a checkerboard flat, and 8.6 % of that parity frame's bytes flip together (the 2 % gate of tests/test_gpu_mammals.py).
constexpr int G_MMA_MIN_RADIUS = 5;

static int pick_seg_h_mma(int n, int H, int W, int d_blocks, int ctas_per_sm) {
    const long strips = (long)((W + G_TW - 1) / G_TW) * n;
    const long slots = (long)sm_count() * ctas_per_sm;
    const int max_segs = std::max(1, H / (2 * M_RB));                 // the score below weighs re-produced rows against wave fill:
                                                                     // a single 1080p frame prefers many short segments, a batch few long ones
    int best = 1;
    double best_score = -1.0;
    for (int segs = 1; segs <= max_segs && segs <= 64; ++segs) {
        int seg_h = (H + segs - 1) / segs;
        seg_h = (seg_h + M_RB - 1) / M_RB * M_RB;
        const long real_segs = (H + seg_h - 1) / seg_h;
        const long ctas = strips * real_segs;
        const long waves = (ctas + slots - 1) / slots;
        const double fill = (double)ctas / (double)(waves * slots);
        const double useful = (double)seg_h / (double)(seg_h + M_RB * d_blocks);
        const double score = fill * useful * (waves >= 2 ? 1.0 : 0.85);
        if (score > best_score + 1e-9) { best_score = score; best = segs; }
    }
    int seg_h = (H + best - 1) / best;
    return (seg_h + M_RB - 1) / M_RB * M_RB;
}

template <int KSH, int D>
static int launch_gauss_mma(const GaussCommon &gc, const DogProducer::Params &pp, const MmaGeom &geo, cudaStream_t st) {
    const size_t smem = (size_t)2 * M_RB * MmaCfg<KSH>::SP * 2 + (size_t)2 * (D + 1) * M_RB * M_HP * 2 +
                        (size_t)M_RB * M_STAGE_PITCH + (size_t)(256 * M_LUT_COPIES + G_ENC_SMEM) * 4 + 2 * (size_t)M_RB * M_RAW_PITCH;
    auto kern = gauss_mma_kernel<KSH, D>;
    AVB_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    dim3 grid((gc.io.W + G_TW - 1) / G_TW, (gc.io.H + gc.seg_h - 1) / gc.seg_h, gc.io.n);
    AVB_TIMED(gc.fixup ? DogProducer::fixup_name() : DogProducer::name(), st);
    kern<<<grid, M_THREADS, smem, st>>>(gc, pp, geo);
    AVB_CUDA_OK(cudaGetLastError());
    return AVB_OK;
}

static int dispatch_gauss_mma(int radius, GaussCommon gc, const DogProducer::Params &q, cudaStream_t st) {
    const int d = radius <= 8 ? 1 : 2;
    MmaGeom geo{};
    geo.radius = radius;
    geo.r4 = (radius + 3) & ~3;
    geo.groups = (G_TW + geo.r4 + radius + 3) / 4;
    geo.div_groups = (65536u + geo.groups - 1) / geo.groups;
    for (int idx = 0; idx < M_RB * geo.groups; ++idx)                        // the multiply-shift division is exact on its range
        if ((int)(((uint32_t)idx * geo.div_groups) >> 16) != idx / geo.groups) { set_error("internal: group divider"); return AVB_E_UNSUPPORTED; }
    gc.radius = radius;
    gc.seg_h = pick_seg_h_mma(gc.io.n, gc.io.H, gc.io.W, d, M_MINB_SINGLE);
    quantize_taps_f16(gc.taps, 2 * radius + 1);
    if (radius <= 8) return launch_gauss_mma<2, 1>(gc, q, geo, st);
    if (radius <= 12) return launch_gauss_mma<2, 2>(gc, q, geo, st);
    return launch_gauss_mma<3, 2>(gc, q, geo, st);
}

static int dispatch_gauss(int radius, GaussCommon &gc, const DogProducer::Params &pp, cudaStream_t st) {
    gc.seg_h = pick_seg_h(gc.io.n, gc.io.H, gc.io.W, radius, radius <= G_MINB3_R ? 3 : G_MINB);
    float Q[6];
    const bool two = rank2_factor(pp.M.m, Q, gc.P);
    DogProducer::Params q = pp;
    if (two) {
        for (int i = 0; i < 6; ++i) q.M.m[i] = Q[i];
        q.M.m[6] = q.M.m[7] = q.M.m[8] = 0.f;
    }
    if (two && radius >= G_MMA_MIN_RADIUS && radius <= 16) return dispatch_gauss_mma(radius, gc, q, st);
    // a rank-2 matrix from G_MMA_MIN_RADIUS up never gets here: no two-plane instantiation for it
    switch (radius) {
#define AVB_CASE(RR) case RR: \
        if constexpr (RR < G_MMA_MIN_RADIUS) if (two) return launch_gauss<RR, 2>(gc, q, st); \
        return launch_gauss<RR, 3>(gc, q, st);
        AVB_CASE(1) AVB_CASE(2) AVB_CASE(3) AVB_CASE(4) AVB_CASE(5) AVB_CASE(6) AVB_CASE(7) AVB_CASE(8)
        AVB_CASE(9) AVB_CASE(10) AVB_CASE(11) AVB_CASE(12) AVB_CASE(13) AVB_CASE(14) AVB_CASE(15) AVB_CASE(16)
#undef AVB_CASE
        default:
            set_error("gaussian radius %d unsupported (ksize must be odd, 3..33)", radius);
            return AVB_E_UNSUPPORTED;
    }
}

static int check_io(const FrameIO &io) {
    if (!io.in || !io.out) { set_error("null frame pointer"); return AVB_E_ARG; }
    if (io.n <= 0 || io.H <= 0 || io.W <= 0) { set_error("bad frame geometry n=%d H=%d W=%d", io.n, io.H, io.W); return AVB_E_ARG; }
    if (io.in_rs < 3LL * io.W || io.out_rs < 3LL * io.W) { set_error("row stride smaller than 3*W"); return AVB_E_ARG; }
    return AVB_OK;
}

}  // namespace avb

using namespace avb;

extern "C" int avb_dichromat_blur_u8(const uint8_t *in, uint8_t *out, int n, int H, int W,
                                     int64_t in_frame_stride, int64_t in_row_stride,
                                     int64_t out_frame_stride, int64_t out_row_stride,
                                     const float *dec_dev, const float *dec_raw_dev, const uint32_t *enc_dev,
                                     const float *m_host, const float *taps_host, int ksize,
                                     int norm_mode, uint32_t *flags_dev, avb_stream_t stream) {
    GaussCommon gc{};
    gc.io = FrameIO{in, out, in_frame_stride, in_row_stride, out_frame_stride, out_row_stride, n, H, W};
    if (int e = check_io(gc.io)) return e;
    AVB_REQUIRE(dec_dev && enc_dev && m_host && taps_host, "null table pointer");
    AVB_REQUIRE(ksize >= 3 && ksize <= G_MAX_TAPS && (ksize & 1), "ksize must be odd, 3..33");
    AVB_REQUIRE(norm_mode == AVB_NORM_DIV255 || (norm_mode == AVB_NORM_AUTO && dec_raw_dev && flags_dev),
                "AVB_NORM_AUTO needs dec_raw_dev and flags_dev");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    for (int i = 0; i < ksize; ++i) gc.taps[i] = taps_host[i];
    gc.enc = enc_dev;
    DogProducer::Params pp{};
    for (int i = 0; i < 9; ++i) pp.M.m[i] = m_host[i];
    pp.lut = dec_dev;
    if (norm_mode == AVB_NORM_AUTO) {
        AVB_CUDA_OK(cudaMemsetAsync(flags_dev, 0, sizeof(uint32_t) * n, st));
        gc.flags = flags_dev;
    }
    gc.fixup = 0;
    if (int e = dispatch_gauss(ksize / 2, gc, pp, st)) return e;
    if (norm_mode == AVB_NORM_AUTO) {
        gc.fixup = 1;
        pp.lut = dec_raw_dev;
        if (int e = dispatch_gauss(ksize / 2, gc, pp, st)) return e;
    }
    return AVB_OK;
}


// ------------------------------------------------------------------------------------ Cat
namespace avb {

// per-frame "some byte >= 2" (the data-dependent branch of get_normalized_image) for kernels that
// do not visit every input pixel themselves.  One byte >= 2 anywhere PROVES the frame maximum is > 1, so the
// question is settled for any ordinary frame by a sparse scan (every row_step-th row: pass 1, 1 / 64 of the
// frame); only a frame without a witness in the sample (all bytes 0 / 1 there) gets the full scan of pass 2,
// whose CTAs leave at once when the flag is already set.  Exact either way; 0.107 -> ~0.01 ms per 20 4K frames.
__global__ void __launch_bounds__(256) frame_flags_kernel(FrameIO io, uint32_t *flags, int row_step, int skip_if_set) {
    const int frame = blockIdx.y;
    if (skip_if_set && flags[frame] != 0) return;
    const uint8_t *src = io.in + (int64_t)frame * io.in_fs;
    const int row_bytes = 3 * io.W;
    uint32_t seen = 0;
    const bool vec = ((io.in_rs & 15) == 0) && ((io.in_fs & 15) == 0) && ((reinterpret_cast<uintptr_t>(io.in) & 15) == 0);
    for (int y = blockIdx.x * row_step; y < io.H; y += gridDim.x * row_step) {
        const uint8_t *row = src + (int64_t)y * io.in_rs;
        int b = 0;
        if (vec) {
            const int nv = row_bytes >> 4;
            for (int i = threadIdx.x; i < nv; i += blockDim.x) {
                const uint4 v = __ldg(reinterpret_cast<const uint4 *>(row) + i);
                seen |= v.x | v.y | v.z | v.w;
            }
            b = nv << 4;
        }
        for (int i = b + threadIdx.x; i < row_bytes; i += blockDim.x) seen |= row[i];
    }
    if (__any_sync(0xffffffffu, (seen & 0xfefefefeu) != 0) && (threadIdx.x & 31) == 0) flags[frame] = 1u;
}

// ------------------------------------------------------------------------------------ cat warp kernel
// Binocular wide-FOV gather + blend + pow decode + 3x3 (animals/cat_widevision_utils.py:46-99, animals/cat.py:95-101)
// -> separable Gaussian -> encode, in the strip / 8-row-block shape of gauss_stream_kernel and with its H pass, V pass
// and encode.  Every map of the warp depends on the column only, so each CTA first turns the per-column tables into
// one record per produced column in shared memory: the live eye view (a single one for every column of the default
// geometry), the byte offset of its left tap, the two bilinear weights and the eye weight, the blend denominator and
// its reciprocal.  A producer task is then one column x 8 rows.  Measured on a B200 at 1000 W, 20 4K frames:
// 1.135 ms with the producer policy of gauss_stream_kernel (tables and tap geometry per 4 rows, both eyes' terms of the
// blend), 0.993 ms here.
//
// cv::remap INTER_LINEAR: map coordinate quantised to 1/32 px, two taps, border constant 0.  A tap outside the
// image gets weight 0 in the record instead of a zeroed sample: both products are +0 (samples are finite and >= 0),
// so the sums are unchanged; its offset is clamped to [-1, W-1] so that it still reads bytes of the staged span.
// A single live eye drops the other eye's terms of the blend: the skipped product is +0 added to a value >= +0.
struct CatParams {
    Mat3 M;             // RGB->LMS, L/M merge, LMS->RGB collapsed into one 3x3 (host, float64 -> f32)
    const float *xl, *xr, *wl, *wr;  // per-column tables, length W (device)
    const float *ws, *rws;           // per column: wl + wr + 1e-8 (float32) and its correctly rounded reciprocal
    const uint32_t *frame_flags;     // per frame: != 0 when some byte >= 2 (written by frame_flags_kernel)
    int norm_mode;                   // AVB_NORM_DIV255: always /255; AVB_NORM_AUTO: /255 iff flag set
};

constexpr int CAT_RAW_PITCH = 960;   // 16 B slack + 58 chunks of 16 B + slack: (128 + 2*16) columns x 2.1 source px x 3 B + alignment slack

// record of one tap pair: {byte offset of the left tap (int bits), weight of the left tap, of the right tap, eye weight}
__device__ __forceinline__ float4 cat_tap(float xs, float w_eye, int W, int &lo, int &hi) {
    const int sx = __float2int_rn(xs * 32.0f);
    const int ix = sx >> 5;
    const float f = (float)(sx & 31) * (1.0f / 32.0f);
    const float w0 = 1.0f - f;
    const int ixc = min(max(ix, -1), W - 1);
    lo = min(lo, ixc);
    hi = max(hi, ixc + 1);
    return make_float4(__int_as_float(3 * ixc), (unsigned)ix < (unsigned)W ? w0 : 0.f, (unsigned)(ix + 1) < (unsigned)W ? f : 0.f, w_eye);
}

// the two taps of one eye view, from a 4-byte aligned row (the shared raw tile, readable a few bytes past either end
// of the span): the two source pixels are 6 contiguous bytes = three 32-bit loads + two funnel shifts
__device__ __forceinline__ void cat_gather_words(const float *norm_s, const uint8_t *q, float w0, float f, float &c0, float &c1, float &c2) {
    const uint32_t *w = reinterpret_cast<const uint32_t *>(reinterpret_cast<uintptr_t>(q) & ~(uintptr_t)3);
    const uint32_t sh = (uint32_t)(reinterpret_cast<uintptr_t>(q) & 3) * 8;
    const uint32_t v0 = w[0], v1 = w[1], v2 = w[2];
    const uint32_t lo = __funnelshift_r(v0, v1, sh), hi = __funnelshift_r(v1, v2, sh);
    const float a0 = norm_s[lo & 0xffu], a1 = norm_s[(lo >> 8) & 0xffu], a2 = norm_s[(lo >> 16) & 0xffu];
    const float b0 = norm_s[lo >> 24], b1 = norm_s[hi & 0xffu], b2 = norm_s[(hi >> 8) & 0xffu];
    c0 = __fadd_rn(__fmul_rn(a0, w0), __fmul_rn(b0, f));
    c1 = __fadd_rn(__fmul_rn(a1, w0), __fmul_rn(b1, f));
    c2 = __fadd_rn(__fmul_rn(a2, w0), __fmul_rn(b2, f));
}
// same from a global row: only taps inside the image (weight != 0) are read
__device__ __forceinline__ void cat_gather_bytes(const float *norm_s, const uint8_t *q, float w0, float f, float &c0, float &c1, float &c2) {
    float a0 = 0.f, a1 = 0.f, a2 = 0.f, b0 = 0.f, b1 = 0.f, b2 = 0.f;
    if (w0 != 0.0f) { a0 = norm_s[q[0]]; a1 = norm_s[q[1]]; a2 = norm_s[q[2]]; }
    if (f != 0.0f) { b0 = norm_s[q[3]]; b1 = norm_s[q[4]]; b2 = norm_s[q[5]]; }
    c0 = __fadd_rn(__fmul_rn(a0, w0), __fmul_rn(b0, f));
    c1 = __fadd_rn(__fmul_rn(a1, w0), __fmul_rn(b1, f));
    c2 = __fadd_rn(__fmul_rn(a2, w0), __fmul_rn(b2, f));
}

__device__ __forceinline__ float cat_decode(float v) {
    // animals/animal_utils.py:5-11 on float32; the power goes through the SFU (ex2(2.4 lg2 x),
    // ~5e-7 relative: far inside the 1-LSB budget of the uint8 result)
    // (arguments stay in [0.09, 1] and exponents in [-8.4, 0]: the .ftz SFU forms are exact enough
    // and need no denormal scaling code around them)
    float l, e;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(l) : "f"((v + 0.055f) * (1.0f / 1.055f)));
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(2.4f * l));
    return v <= 0.04045f ? v * (1.0f / 12.92f) : e;
}

// blend numerators n -> quotient n / (wL + wR + 1e-8), correctly rounded from the per-column reciprocal (one Newton
// step on the quotient) -> decode -> 3x3 (rows 0, 1 of Q in two-plane mode)
__device__ __forceinline__ void cat_finish(const float (&m)[9], float n0, float n1, float n2, float s, float r, float &o0, float &o1, float &o2) {
    float q0 = __fmul_rn(n0, r), q1 = __fmul_rn(n1, r), q2 = __fmul_rn(n2, r);
    q0 = fmaf(fmaf(-q0, s, n0), r, q0);
    q1 = fmaf(fmaf(-q1, s, n1), r, q1);
    q2 = fmaf(fmaf(-q2, s, n2), r, q2);
    const float s0 = cat_decode(__saturatef(q0)), s1 = cat_decode(__saturatef(q1)), s2 = cat_decode(__saturatef(q2));
    o0 = m[0] * s0 + m[1] * s1 + m[2] * s2;
    o1 = m[3] * s0 + m[4] * s1 + m[5] * s2;
    o2 = m[6] * s0 + m[7] * s1 + m[8] * s2;
}

#ifndef CAT_MINB4_R
#define CAT_MINB4_R 4
#endif
// two planes at radius <= 4 (the cat's own 9-tap blur): four CTAs per SM -- 60 registers, no spill, 55 KB of shared
// memory per CTA (CUDA 12.9)
template <int R, int NCH>
struct CatOcc { static constexpr int MIN_BLOCKS = (NCH == 2 && R <= CAT_MINB4_R) ? 4 : GaussOcc<R, NCH>::MIN_BLOCKS; };

template <int R, int NCH>
__global__ void __launch_bounds__(G_THREADS_PER_PLANE * NCH, CatOcc<R, NCH>::MIN_BLOCKS)
cat_warp_kernel(const __grid_constant__ GaussCommon p, const __grid_constant__ CatParams pp) {
    using C = GaussCfg<R>;
    constexpr int THREADS = G_THREADS_PER_PLANE * NCH;
    static_assert(C::IN_W <= THREADS, "one column record per thread");
    extern __shared__ __align__(16) uint8_t smem_raw[];
    float *S = reinterpret_cast<float *>(smem_raw);            // [NCH][RB][S_PITCH] produced rows (+x halo)
    float *X = S + NCH * C::S_PLANE;                           // [NCH][RB][X_PITCH] horizontally blurred rows
    float *Y = X + NCH * C::X_PLANE;                           // [NCH][RB][X_PITCH] fully blurred rows
    float *norm_s = Y + NCH * C::X_PLANE;                      // [256] normalised byte values
    uint32_t *enc_s = reinterpret_cast<uint32_t *>(norm_s + 256);
    float4 *rec_a = reinterpret_cast<float4 *>(enc_s + G_ENC_SMEM);                 // [IN_W] live eye (left eye if both live)
    float4 *rec_b = rec_a + C::IN_W;                                                 // [IN_W] right eye if both live, else weight 0
    float2 *rec_s = reinterpret_cast<float2 *>(rec_b + C::IN_W);                     // [IN_W] blend denominator, its reciprocal
    uint8_t *rawt0 = reinterpret_cast<uint8_t *>(rec_s + C::IN_W);                   // [2][RB][RAW_PITCH] packed input rows (TMA double buffer)
    constexpr int RAW_PITCH = CAT_RAW_PITCH;
    __shared__ __align__(8) uint64_t rbar[2];                                       // completion of the bulk copies of each buffer
    __shared__ int span[3];                                                         // source columns the strip's taps touch: lo, hi; eye mode

    const int frame = blockIdx.z;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int H = p.io.H, W = p.io.W;
    const int x0 = blockIdx.x * G_TW;
    const int y_start = blockIdx.y * p.seg_h;
    const int y_end = min(H, y_start + p.seg_h);
    const uint8_t *src_frame = p.io.in + (int64_t)frame * p.io.in_fs;

    // normalised byte values exactly as NumPy makes them: float32(v) / float32(255), or, when the
    // frame max is <= 1 (get_normalized_image's other branch), the byte itself clipped to [0,1]
    const bool div255 = pp.norm_mode == AVB_NORM_DIV255 || __ldg(pp.frame_flags + frame) != 0;
    for (int i = tid; i < 256; i += THREADS) norm_s[i] = div255 ? __fdiv_rn((float)i, 255.0f) : fminf((float)i, 1.0f);
    copy_to_smem(enc_s, p.enc, min(G_ENC_SMEM, ENC_HEADER + (int)__ldg(p.enc + 2)));
    if (tid == 0) {
        span[0] = 0x7fffffff; span[1] = -1; span[2] = 0;
        gauss_mbar_init(&rbar[0], G_RB);
        gauss_mbar_init(&rbar[1], G_RB);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (tid < C::IN_W) {
        const int x = reflect101(x0 - R + tid, W);
        const float wL = __ldg(pp.wl + x), wR = __ldg(pp.wr + x);
        int lo = 0x7fffffff, hi = -1, mode = 0;
        float4 a = make_float4(0.f, 0.f, 0.f, 0.f), b = a;
        if (wL != 0.0f) { a = cat_tap(__ldg(pp.xl + x), wL, W, lo, hi); mode |= 1; }
        if (wR != 0.0f) {
            const float4 t = cat_tap(__ldg(pp.xr + x), wR, W, lo, hi);
            if (mode) { b = t; mode |= 4; } else { a = t; }
            mode |= 2;
        }
        rec_a[tid] = a;
        rec_b[tid] = b;
        rec_s[tid] = make_float2(__ldg(pp.ws + x), __ldg(pp.rws + x));
        if (mode) { atomicMin(&span[0], lo); atomicMax(&span[1], hi); atomicOr(&span[2], mode); }
    }
    __syncthreads();
    const EncTable enc = enc_view(enc_s);
    uint8_t *dst_frame = p.io.out + (int64_t)frame * p.io.out_fs;

    // a strip outside both eye views (the blind middle third) is identically zero and encodes to byte 0
    if (span[2] == 0) {
        const bool vec_ok = (x0 + G_TW <= W) && ((p.io.out_rs & 15) == 0) && ((p.io.out_fs & 15) == 0) &&
                            ((reinterpret_cast<uintptr_t>(p.io.out) & 15) == 0);
        const int nbytes = min(G_TW, W - x0) * 3;
        for (int y = y_start + warp; y < y_end; y += THREADS / 32) {
            uint8_t *row = dst_frame + (int64_t)y * p.io.out_rs + (int64_t)x0 * 3;
            if (vec_ok) {
                if (lane < G_TW * 3 / 16) reinterpret_cast<uint4 *>(row)[lane] = make_uint4(0u, 0u, 0u, 0u);
            } else {
                for (int b = lane; b < nbytes; b += 32) row[b] = 0;
            }
        }
        return;
    }

    // Raw tile: the packed bytes [a0, a0 + 16*n_chunks) of 8 input rows -- the source columns the strip's taps touch
    // -- fetched with 16-byte loads one block ahead, 16 bytes into each tile row.  Strips with a single live eye view
    // only; the others (and unaligned frames) gather from global memory.
    const bool out4 = ((p.io.out_rs & 3) == 0) && ((p.io.out_fs & 3) == 0) && ((reinterpret_cast<uintptr_t>(p.io.out) & 3) == 0);
    const bool in16 = ((p.io.in_rs & 15) == 0) && ((p.io.in_fs & 15) == 0) && ((reinterpret_cast<uintptr_t>(p.io.in) & 15) == 0);
    const int ixlo = max(span[0], 0), ixhi = min(span[1], W - 1);
    const int a0 = (3 * ixlo) & ~15;
    const int n_chunks = (3 * (ixhi + 1) - a0 + 15) >> 4;
    const bool vec_in = (span[2] == 1 || span[2] == 2) && in16 && n_chunks > 0 && 16 * n_chunks + 32 <= RAW_PITCH &&
                        a0 + 16 * n_chunks <= (int)p.io.in_rs;

    const int n_in_rows = (y_end - y_start) + 2 * R;
    const int n_in_blocks = (n_in_rows + G_RB - 1) / G_RB;

    const int ch = tid >> 7;                         // 128 threads per plane
    const int h_r = tid & 7, h_xg = (tid & 127) >> 3;
    const int v_x = tid & 127;
    float A[2 * R];                                  // partial sums of the 2R output rows in flight
#pragma unroll
    for (int i = 0; i < 2 * R; ++i) A[i] = 0.f;
    float m[9];
#pragma unroll
    for (int i = 0; i < 9; ++i) m[i] = pp.M.m[i];

    auto raw_issue = [&](int yb_, int buf) {
        if (tid < G_RB) {
            const uint8_t *g = src_frame + (int64_t)reflect101(yb_ + tid, H) * p.io.in_rs + a0;
            gauss_bulk_load(rawt0 + buf * (G_RB * RAW_PITCH) + 16 + tid * RAW_PITCH, g, 16u * (uint32_t)n_chunks, &rbar[buf]);
        }
    };
    uint32_t rphase = 0;                             // bit b: parity the next wait on buffer b expects
    if (vec_in) raw_issue(y_start - R, 0);

    auto store = [&](int r, int i, float o0, float o1, float o2) {
        S[0 * C::S_PLANE + r * C::S_PITCH + i] = o0;
        S[1 * C::S_PLANE + r * C::S_PITCH + i] = o1;
        if (NCH == 3) S[2 * C::S_PLANE + r * C::S_PITCH + i] = o2;
    };

    for (int ib = 0; ib < n_in_blocks; ++ib) {
        const int yb = y_start - R + ib * G_RB;      // first input row of this block
        // ---- produce RB rows x IN_W columns of linear-light values: a task is one column x 8 rows
        if (vec_in) {
            // the packed rows of this block were requested one block ahead: wait for the copies, then put
            // the next block's copies in flight (its buffer was last read two barriers ago)
            const int buf = ib & 1;
            gauss_mbar_wait(&rbar[buf], (rphase >> buf) & 1u);
            rphase ^= 1u << buf;
            if (ib + 1 < n_in_blocks) raw_issue(yb + G_RB, buf ^ 1);
            if (tid < C::IN_W) {
                const float4 a = rec_a[tid];
                if (a.w == 0.0f) {                   // outside both eye views: (0*wL + 0*wR)/ws = 0 -> decode(0) = 0
#pragma unroll
                    for (int r = 0; r < G_RB; ++r) store(r, tid, 0.f, 0.f, 0.f);
                } else {
                    const float2 sr = rec_s[tid];
                    const uint8_t *q = rawt0 + buf * (G_RB * RAW_PITCH) + 16 + (__float_as_int(a.x) - a0);
#pragma unroll
                    for (int r = 0; r < G_RB; ++r) {
                        float c0, c1, c2, o0, o1, o2;
                        cat_gather_words(norm_s, q + r * RAW_PITCH, a.y, a.z, c0, c1, c2);
                        cat_finish(m, __fmul_rn(c0, a.w), __fmul_rn(c1, a.w), __fmul_rn(c2, a.w), sr.x, sr.y, o0, o1, o2);
                        store(r, tid, o0, o1, o2);
                    }
                }
            }
        } else {
            // unaligned frames, strips that see both eye views: gather from global memory
            if (tid < C::IN_W) {
                const float4 a = rec_a[tid], b = rec_b[tid];
                const float2 sr = rec_s[tid];
                for (int r = 0; r < G_RB; ++r) {
                    float o0 = 0.f, o1 = 0.f, o2 = 0.f;
                    if (a.w != 0.0f) {
                        const uint8_t *row = src_frame + (int64_t)reflect101(yb + r, H) * p.io.in_rs;
                        float l0, l1, l2;
                        cat_gather_bytes(norm_s, row + __float_as_int(a.x), a.y, a.z, l0, l1, l2);
                        float n0 = __fmul_rn(l0, a.w), n1 = __fmul_rn(l1, a.w), n2 = __fmul_rn(l2, a.w);
                        if (b.w != 0.0f) {
                            float r0, r1, r2;
                            cat_gather_bytes(norm_s, row + __float_as_int(b.x), b.y, b.z, r0, r1, r2);
                            n0 = __fadd_rn(n0, __fmul_rn(r0, b.w));
                            n1 = __fadd_rn(n1, __fmul_rn(r1, b.w));
                            n2 = __fadd_rn(n2, __fmul_rn(r2, b.w));
                        }
                        cat_finish(m, n0, n1, n2, sr.x, sr.y, o0, o1, o2);
                    }
                    store(r, tid, o0, o1, o2);
                }
            }
        }
        __syncthreads();
        gauss_hpass<R>(p, S, X, ch, h_r, h_xg);
        __syncthreads();
        gauss_vpass<R>(p, X, Y, ch, v_x, A);
        __syncthreads();
        gauss_encode_store<R, NCH, THREADS>(p, enc, Y, dst_frame, ib, y_start, y_end, x0, out4);
    }
}

template <int R, int NCH>
static int launch_cat(const GaussCommon &gc, const CatParams &pp, cudaStream_t st) {
    using C = GaussCfg<R>;
    const size_t smem = (size_t)(NCH * C::S_PLANE + 2 * NCH * C::X_PLANE + 256 + G_ENC_SMEM) * 4 + (size_t)C::IN_W * (16 + 16 + 8) +
                        2 * (size_t)G_RB * CAT_RAW_PITCH;
    auto kern = cat_warp_kernel<R, NCH>;
    AVB_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    dim3 grid((gc.io.W + G_TW - 1) / G_TW, (gc.io.H + gc.seg_h - 1) / gc.seg_h, gc.io.n);
    AVB_TIMED("k2_gauss_cat_warp", st);
    kern<<<grid, G_THREADS_PER_PLANE * NCH, smem, st>>>(gc, pp);
    AVB_CUDA_OK(cudaGetLastError());
    return AVB_OK;
}

static int dispatch_cat(int radius, GaussCommon &gc, const CatParams &pp, cudaStream_t st) {
#ifndef G_CAT_SEG_SLOTS
#define G_CAT_SEG_SLOTS 3
#endif
    gc.seg_h = pick_seg_h(gc.io.n, gc.io.H, gc.io.W, radius, radius <= CAT_MINB4_R ? G_CAT_SEG_SLOTS : (radius <= G_MINB3_R ? 3 : G_MINB));
    float Q[6];
    const bool two = rank2_factor(pp.M.m, Q, gc.P);
    CatParams q = pp;
    if (two) {
        for (int i = 0; i < 6; ++i) q.M.m[i] = Q[i];
        q.M.m[6] = q.M.m[7] = q.M.m[8] = 0.f;
    }
    switch (radius) {
#define AVB_CASE(RR) case RR: return two ? launch_cat<RR, 2>(gc, q, st) : launch_cat<RR, 3>(gc, q, st);
        AVB_CASE(1) AVB_CASE(2) AVB_CASE(3) AVB_CASE(4) AVB_CASE(5) AVB_CASE(6) AVB_CASE(7) AVB_CASE(8)
        AVB_CASE(9) AVB_CASE(10) AVB_CASE(11) AVB_CASE(12) AVB_CASE(13) AVB_CASE(14) AVB_CASE(15) AVB_CASE(16)
#undef AVB_CASE
        default:
            set_error("gaussian radius %d unsupported (ksize must be odd, 3..33)", radius);
            return AVB_E_UNSUPPORTED;
    }
}

// Centre zoom (cat_widevision_utils.py:11-29): crop + cv2.resize(INTER_LINEAR) on uint8, restated
// in OpenCV's 11-bit fixed point so the result is bit-exact.  tab = W x int4 {xi0, xi1, xw0, xw1}
// then H x int4 {yi0, yi1, yw0, yw1} (source indices already include the crop origin).
// One thread = 4 consecutive output pixels per row (12 bytes = three 32-bit stores).  The two
// horizontal taps of a pixel are adjacent source pixels (xi1 = xi0 + 1, or xi1 = xi0 with weight 0
// at the right edge), i.e. 6 contiguous bytes: the aligned path fetches them as three 32-bit words
// per source row and realigns with funnel shifts instead of issuing six byte loads.
__device__ __forceinline__ void zoom_taps(const uint32_t *row32, int xi0, int last_word, uint32_t (&a)[3], uint32_t (&b)[3]) {
    const int ob = 3 * xi0, wi = ob >> 2, sh = (ob & 3) * 8;
    const uint32_t w0 = __ldg(row32 + wi), w1 = __ldg(row32 + min(wi + 1, last_word)), w2 = __ldg(row32 + min(wi + 2, last_word));
    const uint32_t lo = __funnelshift_r(w0, w1, sh), hi = __funnelshift_r(w1, w2, sh);
    a[0] = lo & 0xffu; a[1] = (lo >> 8) & 0xffu; a[2] = (lo >> 16) & 0xffu;       // pixel xi0
    b[0] = lo >> 24; b[1] = hi & 0xffu; b[2] = (hi >> 8) & 0xffu;                  // pixel xi0 + 1
}
// cv2.resize is separable: a thread owns 4 output pixels of a column strip and walks down ZOOM_ROWS output
// rows, keeping the horizontally interpolated values (a0*xw0 + a1*xw1, three channels x four pixels) of
// the two source rows in flight in registers.  Going down, the source row pair advances by 0 or 1 per
// output row (scale 1/1.5), so most rows recompute one horizontal row or none instead of two.
#ifndef ZOOM_ROWS_N
#define ZOOM_ROWS_N 32
#endif
constexpr int ZOOM_ROWS = ZOOM_ROWS_N;
#ifndef ZOOM_MINB
// 24 warps per SM (measured, 20 4K frames: 4 -> 0.471 ms, 6 -> 0.406, 8 -> 0.464).  CUDA 12.9 fits it in 80 registers with
// 112 B of spill stores; five CTAs per SM (96 registers, no spill) measured slower on a B200 at 1000 W: 0.437 against 0.409 ms
#define ZOOM_MINB 6
#endif
__global__ void __launch_bounds__(128, ZOOM_MINB) center_zoom_kernel(FrameIO io, const int32_t *__restrict__ tab, int aligned_out, int aligned_in) {
    const int W = io.W, H = io.H;
    const int x4 = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (x4 >= W) return;
    const int y_begin = blockIdx.y * ZOOM_ROWS, y_end = min(H, y_begin + ZOOM_ROWS);
    const uint8_t *src = io.in + (int64_t)blockIdx.z * io.in_fs;
    const int last_word = (3 * W - 1) >> 2;
    const int npx = min(4, W - x4);
    int4 tx[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) tx[j] = __ldg(reinterpret_cast<const int4 *>(tab) + min(x4 + j, W - 1));
    int sa[12], sb[12];                       // (a0*xw0 + a1*xw1) >> 4 of source rows ia, ib
    int ia = -1, ib = -1;
    // the packed words of a source row: three 32-bit words per output pixel hold its two horizontal taps
    // (6 bytes from byte 3*xi0).  Rows are FETCHED one step before they are needed (the next source row is
    // always ib + 1 when upscaling) and only converted when the walk reaches them.
    uint32_t pw[12];
    int pw_row = -2;
    int wi[4], sh[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) { const int ob = 3 * tx[j].x; wi[j] = ob >> 2; sh[j] = (ob & 3) * 8; }
    auto fetch = [&](int r) {
        const uint32_t *row32 = reinterpret_cast<const uint32_t *>(src + (int64_t)r * io.in_rs);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            pw[3 * j] = __ldg(row32 + wi[j]);
            pw[3 * j + 1] = __ldg(row32 + min(wi[j] + 1, last_word));
            pw[3 * j + 2] = __ldg(row32 + min(wi[j] + 2, last_word));
        }
        pw_row = r;
    };
    auto hrow = [&](int r, int (&s)[12]) {
        const uint8_t *row = src + (int64_t)r * io.in_rs;
        if (aligned_in && pw_row != r) fetch(r);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            uint32_t a0[3], a1[3];
            if (aligned_in) {
                const uint32_t lo = __funnelshift_r(pw[3 * j], pw[3 * j + 1], sh[j]), hi = __funnelshift_r(pw[3 * j + 1], pw[3 * j + 2], sh[j]);
                a0[0] = lo & 0xffu; a0[1] = (lo >> 8) & 0xffu; a0[2] = (lo >> 16) & 0xffu;       // pixel xi0
                a1[0] = lo >> 24; a1[1] = hi & 0xffu; a1[2] = (hi >> 8) & 0xffu;                  // pixel xi0 + 1
                // (xi1 == xi0 only where its weight is 0: the neighbour's bytes then multiply 0)
            } else {
#pragma unroll
                for (int c = 0; c < 3; ++c) { a0[c] = row[3 * tx[j].x + c]; a1[c] = row[3 * tx[j].y + c]; }
            }
#pragma unroll
            for (int c = 0; c < 3; ++c) s[3 * j + c] = ((int)a0[c] * tx[j].z + (int)a1[c] * tx[j].w) >> 4;
        }
        if (aligned_in && r + 1 < H) fetch(r + 1);          // the row the walk will need next
    };
    uint8_t *o = io.out + (int64_t)blockIdx.z * io.out_fs + (int64_t)y_begin * io.out_rs + 3 * x4;
    for (int y = y_begin; y < y_end; ++y, o += io.out_rs) {
        const int4 ty = __ldg(reinterpret_cast<const int4 *>(tab) + W + y);      // uniform over the block
        // block-uniform conditions: the empty asm statements keep the compiler from if-converting these
        // bodies into dozens of predicated instructions that would issue on every row
        if (ty.x != ia) {
            asm volatile("");
            if (ty.x == ib) {
#pragma unroll
                for (int i = 0; i < 12; ++i) sa[i] = sb[i];
            } else {
                hrow(ty.x, sa);
            }
            ia = ty.x;
        }
        if (ty.y != ib) {
            asm volatile("");
            if (ty.y == ia) {
#pragma unroll
                for (int i = 0; i < 12; ++i) sb[i] = sa[i];
            } else {
                hrow(ty.y, sb);
            }
            ib = ty.y;
        }
        uint32_t by[12];
#pragma unroll
        for (int i = 0; i < 12; ++i) {
            const int v = ((((ty.z * sa[i]) >> 16) + ((ty.w * sb[i]) >> 16) + 2) >> 2);
            by[i] = (uint32_t)min(255, max(0, v));
        }
        if (aligned_out && npx == 4) {
            uint32_t *o32 = reinterpret_cast<uint32_t *>(o);
#pragma unroll
            for (int q = 0; q < 3; ++q) o32[q] = by[4 * q] | (by[4 * q + 1] << 8) | (by[4 * q + 2] << 16) | (by[4 * q + 3] << 24);
        } else {
            for (int q = 0; q < 3 * npx; ++q) o[q] = (uint8_t)by[q];
        }
    }
}

}  // namespace avb

extern "C" int avb_cat_u8(const uint8_t *in, uint8_t *out_human, uint8_t *out_cat, int n, int H, int W,
                          int64_t in_frame_stride, int64_t in_row_stride,
                          int64_t human_frame_stride, int64_t human_row_stride,
                          int64_t cat_frame_stride, int64_t cat_row_stride,
                          const float *dec_dev, const float *dec_raw_dev,
                          const uint32_t *enc_dev, const float *m_host, const float *taps_host, int ksize,
                          const float *warp_dev, const int32_t *zoom_dev,
                          int norm_mode, uint32_t *flags_dev, avb_stream_t stream) {
    GaussCommon gc{};
    gc.io = FrameIO{in, out_cat, in_frame_stride, in_row_stride, cat_frame_stride, cat_row_stride, n, H, W};
    if (int e = check_io(gc.io)) return e;
    AVB_REQUIRE(enc_dev && m_host && taps_host, "null table pointer");
    AVB_REQUIRE(warp_dev || (dec_dev && (norm_mode == AVB_NORM_DIV255 || dec_raw_dev)), "without warp_dev the decode LUTs are required");
    AVB_REQUIRE(ksize >= 3 && ksize <= G_MAX_TAPS && (ksize & 1), "ksize must be odd, 3..33");
    AVB_REQUIRE(norm_mode == AVB_NORM_DIV255 || (norm_mode == AVB_NORM_AUTO && flags_dev), "AVB_NORM_AUTO needs flags_dev");
    AVB_REQUIRE((out_human == nullptr) == (zoom_dev == nullptr), "out_human and zoom_dev go together");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (norm_mode == AVB_NORM_AUTO && warp_dev) {
        AVB_CUDA_OK(cudaMemsetAsync(flags_dev, 0, sizeof(uint32_t) * n, st));
        AVB_TIMED("frame_flags", st);
        constexpr int STEP = 64;
        const int sampled = (H + STEP - 1) / STEP;
        frame_flags_kernel<<<dim3(sampled < 256 ? sampled : 256, n), 256, 0, st>>>(gc.io, flags_dev, STEP, 0);      // witness search
        frame_flags_kernel<<<dim3(H < 256 ? H : 256, n), 256, 0, st>>>(gc.io, flags_dev, 1, 1);                        // frames still undecided
        AVB_CUDA_OK(cudaGetLastError());
    }
    if (out_human) {
        AVB_REQUIRE(human_row_stride >= 3LL * W, "row stride smaller than 3*W");
        FrameIO zio{in, out_human, in_frame_stride, in_row_stride, human_frame_stride, human_row_stride, n, H, W};
        AVB_REQUIRE(H <= 65535 && n <= 65535, "frame height / batch too large for one launch");
        AVB_REQUIRE((reinterpret_cast<uintptr_t>(zoom_dev) & 15) == 0, "zoom_dev must be 16-byte aligned");
        dim3 grid((W + 511) / 512, (H + ZOOM_ROWS - 1) / ZOOM_ROWS, n);
        const int aligned_out = ((reinterpret_cast<uintptr_t>(out_human) | (uintptr_t)human_frame_stride | (uintptr_t)human_row_stride) & 3) == 0;
        AVB_TIMED("cat_center_zoom", st);
        const int aligned_in = ((reinterpret_cast<uintptr_t>(in) | (uintptr_t)in_frame_stride | (uintptr_t)in_row_stride) & 3) == 0;
        center_zoom_kernel<<<grid, 128, 0, st>>>(zio, zoom_dev, aligned_out, aligned_in);
        AVB_CUDA_OK(cudaGetLastError());
    }
    for (int i = 0; i < ksize; ++i) gc.taps[i] = taps_host[i];
    gc.enc = enc_dev;
    if (!warp_dev) {
        // ENABLE_FOV_WARP = False (cat.py:21, :84): no gather, so the input is plain uint8 and the
        // LUT producer applies -- decode -> collapsed L/M-merge matrix -> blur -> float64-tail encode
        DogProducer::Params dp{};
        for (int i = 0; i < 9; ++i) dp.M.m[i] = m_host[i];
        dp.lut = dec_dev;
        if (norm_mode == AVB_NORM_AUTO) {
            AVB_CUDA_OK(cudaMemsetAsync(flags_dev, 0, sizeof(uint32_t) * n, st));
            gc.flags = flags_dev;
        }
        gc.fixup = 0;
        if (int e = dispatch_gauss(ksize / 2, gc, dp, st)) return e;
        if (norm_mode == AVB_NORM_AUTO) {
            gc.fixup = 1;
            dp.lut = dec_raw_dev;
            if (int e = dispatch_gauss(ksize / 2, gc, dp, st)) return e;
        }
        return AVB_OK;
    }
    gc.flags = nullptr;   // the warp does not see every pixel: normalisation comes from frame_flags_kernel
    gc.fixup = 0;
    CatParams pp{};
    for (int i = 0; i < 9; ++i) pp.M.m[i] = m_host[i];
    pp.xl = warp_dev; pp.xr = warp_dev + W; pp.wl = warp_dev + 2 * W; pp.wr = warp_dev + 3 * W;
    pp.ws = warp_dev + 4 * W; pp.rws = warp_dev + 5 * W;
    pp.frame_flags = flags_dev;
    pp.norm_mode = norm_mode;
    return dispatch_cat(ksize / 2, gc, pp, st);
}
