// K4: MST++ RGB -> 31-band hyperspectral inference (reference
// ml/MST_plus_plus/predict_code/architecture/MST_Plus_Plus.py:88-293), the one dense contraction on
// the hot path.
//
// Layout: every feature map is channels-last [B, H, W, Cp] with the channel count padded to a
// multiple of 32 (31 -> 32, 62 -> 64, 124 -> 128; FFN hidden 124/248/496 -> 128/256/512); padded
// channels are exactly zero everywhere (weights are zero padded), so they never leak.  The residual
// stream, LayerNorm, q/k norms, the spectral Gram matrix and the softmax stay fp32; GEMM operands
// are bf16 with fp32 accumulation (SURVEY.md 8a-19: the 1e-2 budget needs exactly that split).
//
// Every convolution / linear layer is one implicit GEMM  Y[pixels, Cout] = gather(X)[pixels, K] W^T
// through a single kernel template (pointwise, two-source concat, 3x3, 4x4 stride 2; the 2x2
// transposed conv is a pointwise GEMM with a pixel-shuffle store).  The spectral attention
// (MS_MSA, :110-139) is algebraically folded: softmax(rescale * K_hat Q_hat^T) is a 31x31 matrix
// per head that depends on ALL pixels, so each layer is two-phase --
//   phase 1  q,k,v = x Wqkv^T (one GEMM), Gram + norms reduced over all pixels (fp32 atomics)
//   phase 2  M = Wproj . blockdiag(attn)  (c x c, per image), out = v M^T + b + pos_emb(v) + x
// -- i.e. attention-apply and the output projection become ONE pointwise GEMM on v.
#include <cuda.h>          // CUtensorMap and its enums only: cuTensorMapEncodeTiled is fetched through the runtime
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <cstdlib>
#include <vector>

#include "avb_common.cuh"

namespace avb {
namespace k4 {

typedef __nv_bfloat16 bf16;

constexpr int NF = 31;                 // n_feat = dim_head
constexpr int64_t N_PARAMS = 1619625;  // MST_Plus_Plus().state_dict() element count

static inline int pad32(int c) { return (c + 31) / 32 * 32; }

// GELU with the exact-erf definition of the reference (MST_Plus_Plus.py:68-70, F.gelu default):
//   gelu(x) = x Phi(x) = max(x, 0) - |x| h,   h = erfc(|x| / sqrt 2) / 2,
// erfc through Abramowitz & Stegun 7.1.26 on the SFU (one rcp, one ex2): |error| < 2e-7 absolute and no
// cancellation on either side of zero -- far inside the bf16 rounding of every tensor this feeds -- in
// 14 instructions (erff() takes about 40).  The argument is pre-scaled by sqrt(log2 e) so that
// exp(-z^2) is a bare ex2 of -(a*a).
__device__ __forceinline__ float gelu(float x) {
    constexpr float S = 1.2011224087864498f;                   // sqrt(log2 e)
    const float a = fabsf(x) * (0.70710678118654752f * S);
    float t, e;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t) : "f"(fmaf(0.3275911f / S, a, 1.0f)));
    float p = 0.5f * 1.061405429f;
    p = fmaf(p, t, 0.5f * -1.453152027f);
    p = fmaf(p, t, 0.5f * 1.421413741f);
    p = fmaf(p, t, 0.5f * -0.284496736f);
    p = fmaf(p, t, 0.5f * 0.254829592f);
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(-(a * a)));
    const float h = (p * t) * e;
    return fmaf(-fabsf(x), h, fmaxf(x, 0.0f));
}

// ------------------------------------------------------------------------------------ programmatic dependent launch
// The forward is a chain of ~160 short dependent kernels.  Every kernel starts with pdl_wait() --
// griddepcontrol.wait: the preceding kernel has completed and its writes are visible -- and is
// launched with programmatic stream serialization, so its launch latency and CTA ramp-up overlap
// the tail of its predecessor instead of adding to it.
__device__ __forceinline__ void pdl_wait() {
    asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}
template <typename P>
static void launch_pdl(void (*kern)(P), dim3 grid, dim3 block, size_t smem, cudaStream_t st, const P &p) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    cudaLaunchKernelEx(&cfg, kern, p);
}

// ------------------------------------------------------------------------------------ implicit GEMM
constexpr int BM = 128, BK = 32;
constexpr int GEMM_THREADS = 256;

enum { MODE_PW = 0, MODE_C3 = 1, MODE_C4S2 = 2 };
enum { OUT_ROWS = 0, OUT_CONVT = 1, OUT_CROP = 2 };

struct GemmP {
    const void *A1, *A2;       // MODE_PW: [B*rows, lda]; conv modes: feature map [B, Hi, Wi, lda1]
    int lda1, lda2, K1, K;     // K1: extent of K taken from A1 (the rest from A2), K multiple of 32
    const bf16 *W;             // [Np][K] row-major (k contiguous)
    const float *W32;          // the same matrix in fp32 (tf32 TMA kernel only)
    long long w_bstride;       // element stride between batch items (0: shared weights)
    int Np;
    int rows;                  // output rows (pixels) per batch item
    int Hi, Wi, Ho, Wo, Cpin;  // conv geometry
    const float *bias;         // [Np] or null
    const float *res1; int ldr1;   // fp32 residual, row-indexed like the output rows
    const bf16 *res2; int ldr2;    // bf16 residual
    int gelu;
    void *out; int ldo; int out_bf16;
    int out_mode;
    int Hreal, Wreal, Cpo, crop_top, crop_left;   // OUT_CONVT: Cpo; OUT_CROP: real size + crop origin
    float *zero_ptr; int zero_n;                  // pointwise pipeline only: block (0,0,0) clears this buffer (attention statistics)
    const float *ln_g, *ln_b; int ln_c;           // pointwise pipeline only: LayerNorm over the ln_c real channels of the fp32 A rows
    // OUT_CROP only (conv_out): band projection fused on the output -- bands_out[px][r] += sum_c v[c] * band_w[r][c]
    // (uv_helpers.py:142-146 integrate_band on the network's cube; mantis_shrimp.py:49-60).  out may then be null.
    const float *band_w; float *bands_out; int n_bands;
};

__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
    __nv_bfloat162 t = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t *>(&t);
}

// ------------------------------------------------------------------------------------ tcgen05 implicit GEMM
// One CTA: 128 output rows x BN output channels, K streamed in chunks of 32 through a two-stage
// shared-memory ring (global loads of chunk i+1 are in flight while chunk i feeds the tensor cores).
// The contraction runs on the 5th-generation tensor cores: one elected thread issues tcgen05.mma (M = 128 rows, N = BN, K = 16
// per instruction) on shared-memory operands described by UMMA descriptors, the fp32 accumulator
// lives in TMEM (BN columns x 128 lanes) and comes back through tcgen05.ld for the epilogue.
//
// Operand layout in shared memory: canonical K-major, no swizzle -- 8x8 "core matrices" (8 rows x
// 16 bytes, rows 16 B apart) tiled  [k-chunk of 8][row-block of 8]:
//     offset(row, kchunk) = kchunk * LBO + (row / 8) * 128 + (row % 8) * 16,   SBO = 128 B,
//     LBO = (rows / 8) * 128 B.
// The loaders are ordinary threads (they convert fp32 -> bf16 and do the conv gathers), so each
// stage is published to the async proxy with fence.proxy.async before the MMA is issued; a stage
// is recycled when the tcgen05.commit mbarrier of the MMAs that read it has completed.
namespace tc {

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    const uint32_t a = smem_u32(bar);
    uint32_t ok = 0;
    while (!ok) {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(ok) : "r"(a), "r"(parity) : "memory");
    }
}
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    // cute::UMMA::SmemDescriptor: start [0,14), LBO [16,30), SBO [32,46) (all >> 4), version = 1 at
    // [46,48), layout type SWIZZLE_NONE = 0 at [61,64)
    return (uint64_t)((saddr & 0x3ffffu) >> 4) | ((uint64_t)(lbo_bytes >> 4) << 16) | ((uint64_t)(sbo_bytes >> 4) << 32) | (1ull << 46);
}
__device__ __forceinline__ void mma_f16(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
                 ::"r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void mma_tf32(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
                 ::"r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void mma_commit(uint64_t *bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16]) {
    uint32_t r[16];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                   "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
                 : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}

// Epilogue of one 128 x BN accumulator tile: warp w owns TMEM lanes 32*(w%4).. (rows) and column half
// w/4; bias, GELU, fp32 / bf16 residuals and the three store modes are fused here.
enum { EPI_BIAS = 1, EPI_GELU = 2, EPI_RES1 = 4, EPI_RES2 = 8, EPI_OUTBF16 = 16, EPI_CONVT = 32, EPI_RUNTIME = -1 };
// flag word of a parameter block (what a compile-time EPI must equal for the specialised kernels)
static inline int epi_of(const GemmP &p) {
    return (p.bias ? EPI_BIAS : 0) | (p.gelu ? EPI_GELU : 0) | (p.res1 ? EPI_RES1 : 0) | (p.res2 ? EPI_RES2 : 0) |
           (p.out_bf16 ? EPI_OUTBF16 : 0) | (p.out_mode == OUT_CONVT ? EPI_CONVT : 0);
}

// PRE: the residual rows were prefetched into registers by the caller (pre1: fp32, BN/8 vectors per
// thread; pre2: bf16, BN/16 vectors) instead of being loaded -- and waited for -- inside the epilogue.
template <int BN, int EPI, bool PRE = false>
__device__ __forceinline__ void epilogue_tile(const GemmP &p, uint32_t tmem_d, int b, int m_base, int n_base, int warp, int lane,
                                              const uint4 *pre1 = nullptr, const uint4 *pre2 = nullptr) {
    constexpr bool RT = EPI == EPI_RUNTIME;
    const bool has_bias = RT ? p.bias != nullptr : (EPI & EPI_BIAS) != 0, has_gelu = RT ? p.gelu != 0 : (EPI & EPI_GELU) != 0;
    const bool has_res1 = RT ? p.res1 != nullptr : (EPI & EPI_RES1) != 0, has_res2 = RT ? p.res2 != nullptr : (EPI & EPI_RES2) != 0;
    const bool out_bf16 = RT ? p.out_bf16 != 0 : (EPI & EPI_OUTBF16) != 0;
    const int out_mode = RT ? p.out_mode : ((EPI & EPI_CONVT) ? OUT_CONVT : OUT_ROWS);
    constexpr int HALF = BN / 2;
    const int m = m_base + 32 * (warp & 3) + lane;
    const int col0 = (warp >> 2) * HALF;
    const long long row = (long long)b * p.rows + m;
    long long obase = 0;
    int cy = 0, cx = 0;
    bool crop_ok = true;
    if (out_mode == OUT_ROWS) obase = row * p.ldo;
    else { cy = m / p.Wo; cx = m - cy * p.Wo; }
    if (out_mode == OUT_CROP) {
        cy -= p.crop_top; cx -= p.crop_left;
        crop_ok = (unsigned)cy < (unsigned)p.Hreal && (unsigned)cx < (unsigned)p.Wreal;
        obase = (((long long)b * p.Hreal + cy) * p.Wreal + cx) * NF;
    }
#pragma unroll (PRE ? 4 : 2)
    for (int c = 0; c < HALF; c += 16) {
        float v[16];
        tmem_ld16(tmem_d + ((uint32_t)(32 * (warp & 3)) << 16) + (uint32_t)(col0 + c), v);     // all lanes: .sync.aligned
        if (m < p.rows) {
            const int n0 = n_base + col0 + c;
#pragma unroll
            for (int i = 0; i < 16; ++i) {
                if (has_bias) v[i] += __ldg(p.bias + n0 + i);
                if (has_gelu) v[i] = gelu(v[i]);
            }
            if (has_res1) {
#pragma unroll
                for (int i = 0; i < 16; i += 4) {
                    const float4 r = PRE ? *reinterpret_cast<const float4 *>(&pre1[(c + i) / 4])
                                         : *reinterpret_cast<const float4 *>(p.res1 + row * p.ldr1 + n0 + i);
                    v[i] += r.x; v[i + 1] += r.y; v[i + 2] += r.z; v[i + 3] += r.w;
                }
            }
            if (has_res2) {
#pragma unroll
                for (int i = 0; i < 16; i += 8) {
                    const uint4 raw = PRE ? pre2[(c + i) / 8] : *reinterpret_cast<const uint4 *>(p.res2 + row * p.ldr2 + n0 + i);
                    const __nv_bfloat162 *h2 = reinterpret_cast<const __nv_bfloat162 *>(&raw);
#pragma unroll
                    for (int q = 0; q < 4; ++q) { v[i + 2 * q] += __low2float(h2[q]); v[i + 2 * q + 1] += __high2float(h2[q]); }
                }
            }
            if (out_mode == OUT_ROWS) {
                if (out_bf16) {
#pragma unroll
                    for (int i = 0; i < 16; i += 8)
                        *reinterpret_cast<uint4 *>((bf16 *)p.out + obase + n0 + i) =
                            make_uint4(pack_bf16(v[i], v[i + 1]), pack_bf16(v[i + 2], v[i + 3]), pack_bf16(v[i + 4], v[i + 5]), pack_bf16(v[i + 6], v[i + 7]));
                } else {
#pragma unroll
                    for (int i = 0; i < 16; i += 4)
                        *reinterpret_cast<float4 *>((float *)p.out + obase + n0 + i) = make_float4(v[i], v[i + 1], v[i + 2], v[i + 3]);
                }
            } else if (out_mode == OUT_CONVT) {
                const int q = n0 / p.Cpo, co = n0 - q * p.Cpo;       // 16-column groups never straddle a (dy,dx) block
                const long long o = ((((long long)b * 2 * p.Ho) + 2 * cy + (q >> 1)) * (2 * p.Wo) + 2 * cx + (q & 1)) * p.ldo + co;
#pragma unroll
                for (int i = 0; i < 16; i += 4)
                    *reinterpret_cast<float4 *>((float *)p.out + o + i) = make_float4(v[i], v[i + 1], v[i + 2], v[i + 3]);
            } else if (crop_ok) {
                if (p.out != nullptr) {
#pragma unroll
                    for (int i = 0; i < 16; ++i)
                        if (n0 + i < NF) ((float *)p.out)[obase + n0 + i] = v[i];
                }
                if (p.bands_out != nullptr) {
                    // a pixel's 32 channels sit in two threads (16 each): both add their half into the zero-initialised
                    // band map; a two-term sum does not depend on the order of the additions, so this stays reproducible
                    float *bo = p.bands_out + (obase / NF) * p.n_bands;
                    for (int r = 0; r < p.n_bands; ++r) {
                        const float *w = p.band_w + r * NF + n0;
                        float acc = 0.f;
#pragma unroll
                        for (int i = 0; i < 16; ++i)
                            if (n0 + i < NF) acc = fmaf(v[i], __ldg(w + i), acc);
                        atomicAdd(bo + r, acc);
                    }
                }
            }
        }
    }
}

template <int BN, bool A_BF16, int MODE, bool DEEP>
__global__ void __launch_bounds__(GEMM_THREADS) gemm_tc_kernel(const __grid_constant__ GemmP p) {
    pdl_wait();
    constexpr int A_LBO = (BM / 8) * 128, B_LBO = (BN / 8) * 128;        // bytes between k-chunks of 8
    constexpr int A_STAGE = (BK / 8) * A_LBO, B_STAGE = (BK / 8) * B_LBO;
    constexpr int TMEM_COLS = BN <= 32 ? 32 : (BN <= 64 ? 64 : (BN <= 128 ? 128 : 256));     // power of two >= BN
    extern __shared__ __align__(1024) uint8_t dsm[];
    uint8_t (*As)[A_STAGE] = reinterpret_cast<uint8_t (*)[A_STAGE]>(dsm);                  // [2][A_STAGE]
    uint8_t (*Bs)[B_STAGE] = reinterpret_cast<uint8_t (*)[B_STAGE]>(dsm + 2 * A_STAGE);    // [2][B_STAGE]
    __shared__ __align__(8) uint64_t mbar[2];
    __shared__ uint32_t tmem_base_s;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int b = blockIdx.z;
    const int m_base = blockIdx.x * BM, n_base = blockIdx.y * BN;

    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_s)), "n"(TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    if (tid == 32) {
        mbar_init(&mbar[0], 1);
        mbar_init(&mbar[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }

    // ---- A loader: thread -> (row, 16-wide half of the 32-wide chunk)
    const int lr = tid >> 1, lh = tid & 1;
    const int lm = m_base + lr;
    const bool row_ok = lm < p.rows;
    int oy = 0, ox = 0;
    if (MODE != MODE_PW) { oy = lm / p.Wo; ox = lm - oy * p.Wo; }
    auto a_src = [&](int kbase, bool &ok) -> const void * {
        ok = row_ok;
        if (MODE == MODE_PW) {
            const long long row = (long long)b * p.rows + lm;
            if (kbase < p.K1) {
                const long long off = row * p.lda1 + kbase + 16 * lh;
                return A_BF16 ? (const void *)((const bf16 *)p.A1 + off) : (const void *)((const float *)p.A1 + off);
            }
            const long long off = row * p.lda2 + (kbase - p.K1) + 16 * lh;
            return A_BF16 ? (const void *)((const bf16 *)p.A2 + off) : (const void *)((const float *)p.A2 + off);
        }
        const int tap = kbase / p.Cpin, c0 = kbase - tap * p.Cpin;
        int yy, xx;
        if (MODE == MODE_C3) { yy = oy + tap / 3 - 1; xx = ox + tap % 3 - 1; }
        else { yy = 2 * oy - 1 + (tap >> 2); xx = 2 * ox - 1 + (tap & 3); }
        ok = row_ok && (unsigned)yy < (unsigned)p.Hi && (unsigned)xx < (unsigned)p.Wi;
        const long long off = (((long long)b * p.Hi + yy) * p.Wi + xx) * p.lda1 + c0 + 16 * lh;
        return A_BF16 ? (const void *)((const bf16 *)p.A1 + off) : (const void *)((const float *)p.A1 + off);
    };
    // Register ring: the global loads of chunk kc + D are issued while chunk kc feeds the tensor cores, so
    // the K loop pays the L2 / HBM latency once per D chunks instead of once per chunk (the conv layers
    // have 9 .. 32 chunks and, at the coarse levels, fewer CTAs than SMs to hide it otherwise; DEEP is chosen
    // for those -- grids of several waves hide the latency with resident CTAs and prefer the registers).  Rows are
    // kept RAW in the ring (fp32 rows are converted when they are stored to shared memory) so that
    // nothing waits on a load before its turn.
    constexpr int B_PER_THREAD = (BN * 4 + GEMM_THREADS - 1) / GEMM_THREADS;
    constexpr int A_VEC = A_BF16 ? 2 : 4;
    constexpr int D = !DEEP ? 1 : ((A_VEC + B_PER_THREAD) <= 5 ? 4 : ((A_VEC + B_PER_THREAD) <= 6 ? 3 : 2));
    uint4 araw[D][A_VEC];
    uint4 breg[D][B_PER_THREAD];
    const bf16 *Wb = p.W + (long long)b * p.w_bstride;
    auto fetch = [&](int kc, uint4 (&ar)[A_VEC], uint4 (&br)[B_PER_THREAD]) {
        const int kbase = kc * BK;
        bool ok;
        const uint4 *src = reinterpret_cast<const uint4 *>(a_src(kbase, ok));
#pragma unroll
        for (int i = 0; i < A_VEC; ++i) ar[i] = ok ? __ldg(src + i) : make_uint4(0u, 0u, 0u, 0u);
#pragma unroll
        for (int i = 0; i < B_PER_THREAD; ++i) {
            const int idx = tid + i * GEMM_THREADS;
            if (idx < BN * 4) {
                const int n = idx >> 2, q = idx & 3;
                br[i] = __ldg(reinterpret_cast<const uint4 *>(Wb + (long long)(n_base + n) * p.K + kbase) + q);
            }
        }
    };
    auto store = [&](int st, const uint4 (&ar)[A_VEC], const uint4 (&br)[B_PER_THREAD]) {
        uint8_t *d = &As[st][(2 * lh) * A_LBO + (lr >> 3) * 128 + (lr & 7) * 16];      // k-chunks 2*lh and 2*lh+1 of row lr
        if (A_BF16) {
            *reinterpret_cast<uint4 *>(d) = ar[0];
            *reinterpret_cast<uint4 *>(d + A_LBO) = ar[1];
        } else {
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const float4 f0 = *reinterpret_cast<const float4 *>(&ar[2 * h]), f1 = *reinterpret_cast<const float4 *>(&ar[2 * h + 1]);
                *reinterpret_cast<uint4 *>(d + h * A_LBO) =
                    make_uint4(pack_bf16(f0.x, f0.y), pack_bf16(f0.z, f0.w), pack_bf16(f1.x, f1.y), pack_bf16(f1.z, f1.w));
            }
        }
#pragma unroll
        for (int i = 0; i < B_PER_THREAD; ++i) {
            const int idx = tid + i * GEMM_THREADS;
            if (idx < BN * 4) {
                const int n = idx >> 2, q = idx & 3;
                *reinterpret_cast<uint4 *>(&Bs[st][q * B_LBO + (n >> 3) * 128 + (n & 7) * 16]) = br[i];
            }
        }
    };

    const int nk = p.K / BK;
#pragma unroll
    for (int u = 0; u < D; ++u)
        if (u < nk) fetch(u, araw[u], breg[u]);
    store(0, araw[0], breg[0]);
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_d = tmem_base_s;
    // instruction descriptor (cute::UMMA::InstrDescriptor): D = F32, A = B = BF16, both K-major
    constexpr uint32_t IDESC = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);

    for (int kc0 = 0; kc0 < nk; kc0 += D) {
#pragma unroll
        for (int u = 0; u < D; ++u) {           // ring slot of chunk kc is kc % D = u (static)
            const int kc = kc0 + u;
            if (kc < nk) {
                const int st = kc & 1;
                if (D == 1 && kc + 1 < nk) fetch(kc + 1, araw[0], breg[0]);      // single slot: it was stored last iteration
                if (tid == 0) {
                    tc_fence_after();
                    const uint32_t a0 = smem_u32(&As[st][0]), b0 = smem_u32(&Bs[st][0]);
#pragma unroll
                    for (int j = 0; j < BK / 16; ++j)
                        mma_f16(tmem_d, make_desc(a0 + 2 * j * A_LBO, A_LBO, 128), make_desc(b0 + 2 * j * B_LBO, B_LBO, 128), IDESC,
                                (kc > 0 || j > 0) ? 1u : 0u);
                    mma_commit(&mbar[st]);          // arrives when every MMA issued so far has finished reading smem
                }
                if (kc + 1 < nk) {
                    if (kc >= 1) mbar_wait(&mbar[st ^ 1], (uint32_t)(((kc - 1) >> 1) & 1));    // chunk kc-1 done with stage st^1
                    store(st ^ 1, araw[(u + 1) % D], breg[(u + 1) % D]);
                    fence_async_smem();
                }
                if (D > 1 && kc + D < nk) fetch(kc + D, araw[u], breg[u]);       // slot u was drained by the store of the previous iteration
                __syncthreads();
            }
        }
    }
    mbar_wait(&mbar[(nk - 1) & 1], (uint32_t)(((nk - 1) >> 1) & 1));
    tc_fence_after();

    epilogue_tile<BN, EPI_RUNTIME>(p, tmem_d, b, m_base, n_base, warp, lane);
    tc_fence_before();
    __syncthreads();
    if (warp == 0) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_d), "n"(TMEM_COLS) : "memory");
    }
}

// ------------------------------------------------------------------------------------ pointwise pipeline
// Pointwise GEMMs (q|k|v, attention projection, FFN in / out, transposed conv, skip fusion) with
// K <= 128: the CTA keeps its weight tile resident in shared memory and walks over a strided
// sequence of 128-row tiles as a software pipeline --
//     global loads of tile i+2 (registers)  ||  tcgen05.mma of tile i+1 (TMEM buffer (i+1)&1)  ||  epilogue of tile i
// -- so neither the HBM/L2 latency of the A rows nor the tensor-core latency is exposed, and one
// __syncthreads per tile is all the CTA-wide synchronisation there is.  The whole K extent of a
// tile sits in one shared-memory stage (two stages), the accumulator is double buffered in TMEM.
// Optional fused LayerNorm (PreNorm in front of the FFN, MST_Plus_Plus.py:57-65): the two loader
// threads of a row hold all its channels, so mean / variance are one shuffle away and the
// normalised bf16 row goes straight into the operand tile -- no LayerNorm launch, no bf16 copy of x.
template <int BN, int KP, bool A_BF16, bool LN, int EPI>
__global__ void __launch_bounds__(GEMM_THREADS) gemm_pw_kernel(const __grid_constant__ GemmP p) {
    pdl_wait();
    static_assert(!(LN && A_BF16), "LayerNorm is fused on the fp32 residual stream");
    constexpr int A_LBO = (BM / 8) * 128, B_LBO = (BN / 8) * 128;
    constexpr int A_STAGE = (KP / 8) * A_LBO, B_BYTES = (KP / 8) * B_LBO;
    constexpr int TMEM_COLS = 2 * BN <= 32 ? 32 : (2 * BN <= 64 ? 64 : (2 * BN <= 128 ? 128 : (2 * BN <= 256 ? 256 : 512)));
    constexpr int BUF1 = TMEM_COLS / 2;                       // column offset of the second accumulator
    constexpr int CPT = KP / 2;                               // channels per loader thread (two threads per row)
    constexpr int NV = A_BF16 ? CPT / 8 : CPT / 4;            // 16-byte vectors per loader thread
    extern __shared__ __align__(1024) uint8_t dsm[];
    uint8_t *As = dsm;                                        // [2][A_STAGE]
    uint8_t *Bs = dsm + 2 * A_STAGE;                          // [B_BYTES]
    float *ln_s = reinterpret_cast<float *>(dsm + 2 * A_STAGE + B_BYTES);      // gamma[KP] | beta[KP]
    __shared__ __align__(8) uint64_t mbar[2];
    __shared__ uint32_t tmem_base_s;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int b = blockIdx.z, n_base = blockIdx.y * BN;
    const int m_tiles = (p.rows + BM - 1) / BM;
    const int n_my = ((int)blockIdx.x < m_tiles) ? (m_tiles - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;

    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_s)), "n"(TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    if (tid == 32) {
        mbar_init(&mbar[0], 1);
        mbar_init(&mbar[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (p.zero_ptr && blockIdx.x == 0 && blockIdx.y == 0 && blockIdx.z == 0)
        for (int i = tid; i < p.zero_n; i += GEMM_THREADS) p.zero_ptr[i] = 0.f;
    {   // resident weight tile: BN rows x KP, canonical K-major
        const bf16 *Wb = p.W + (long long)b * p.w_bstride;
        constexpr int NVEC = BN * (KP / 8), BATCH = 8;                 // eight 16-byte loads in flight per thread
        for (int i0 = 0; i0 < NVEC; i0 += BATCH * GEMM_THREADS) {
            uint4 wv[BATCH];
#pragma unroll
            for (int u = 0; u < BATCH; ++u) {
                const int idx = i0 + u * GEMM_THREADS + tid;
                if (idx < NVEC) {
                    const int n = idx / (KP / 8), q = idx - n * (KP / 8);
                    wv[u] = __ldg(reinterpret_cast<const uint4 *>(Wb + (long long)(n_base + n) * p.K) + q);
                }
            }
#pragma unroll
            for (int u = 0; u < BATCH; ++u) {
                const int idx = i0 + u * GEMM_THREADS + tid;
                if (idx < NVEC) {
                    const int n = idx / (KP / 8), q = idx - n * (KP / 8);
                    *reinterpret_cast<uint4 *>(Bs + q * B_LBO + (n >> 3) * 128 + (n & 7) * 16) = wv[u];
                }
            }
        }
        if (LN) {
            for (int i = tid; i < KP; i += GEMM_THREADS) {
                ln_s[i] = i < p.ln_c ? __ldg(p.ln_g + i) : 0.f;
                ln_s[KP + i] = i < p.ln_c ? __ldg(p.ln_b + i) : 0.f;
            }
        }
    }

    // ---- A loader: thread -> (row, half of the K extent); a two-source GEMM (cat([up, skip])) takes
    // half 0 from A1 and half 1 from A2
    const int lr = tid >> 1, lh = tid & 1;
    const bool two = p.K1 < p.K;
    const uint8_t *abase = static_cast<const uint8_t *>((two && lh) ? p.A2 : p.A1);
    const long long a_ld = (two && lh) ? p.lda2 : p.lda1;
    const int a_c0 = two ? 0 : lh * CPT;
    uint4 areg[NV];
    auto a_fetch = [&](int tile) {
        const int lm = tile * BM + lr;
        if (lm < p.rows) {
            const long long off = ((long long)b * p.rows + lm) * a_ld + a_c0;
            const uint4 *q = reinterpret_cast<const uint4 *>(abase + off * (A_BF16 ? 2 : 4));
#pragma unroll
            for (int i = 0; i < NV; ++i) areg[i] = __ldg(q + i);
        } else {
#pragma unroll
            for (int i = 0; i < NV; ++i) areg[i] = make_uint4(0u, 0u, 0u, 0u);
        }
    };
    auto a_store = [&](int st) {
        uint8_t *d = As + st * A_STAGE + (lh * (CPT / 8)) * A_LBO + (lr >> 3) * 128 + (lr & 7) * 16;
        if (A_BF16) {
#pragma unroll
            for (int i = 0; i < NV; ++i) *reinterpret_cast<uint4 *>(d + i * A_LBO) = areg[i];
        } else {
            float mean = 0.f, rstd = 1.f;
            if (LN) {
                const int ch0 = lh * CPT;
                float s = 0.f;
#pragma unroll
                for (int i = 0; i < NV; ++i) {
                    const float4 f = *reinterpret_cast<const float4 *>(&areg[i]);
                    s += (ch0 + 4 * i < p.ln_c ? f.x : 0.f) + (ch0 + 4 * i + 1 < p.ln_c ? f.y : 0.f) +
                         (ch0 + 4 * i + 2 < p.ln_c ? f.z : 0.f) + (ch0 + 4 * i + 3 < p.ln_c ? f.w : 0.f);
                }
                s += __shfl_xor_sync(0xffffffffu, s, 1);
                mean = s / (float)p.ln_c;
                float q = 0.f;
#pragma unroll
                for (int i = 0; i < NV; ++i) {
                    const float4 f = *reinterpret_cast<const float4 *>(&areg[i]);
                    const float d0 = ch0 + 4 * i < p.ln_c ? f.x - mean : 0.f, d1 = ch0 + 4 * i + 1 < p.ln_c ? f.y - mean : 0.f;
                    const float d2 = ch0 + 4 * i + 2 < p.ln_c ? f.z - mean : 0.f, d3 = ch0 + 4 * i + 3 < p.ln_c ? f.w - mean : 0.f;
                    q += d0 * d0 + d1 * d1 + d2 * d2 + d3 * d3;
                }
                q += __shfl_xor_sync(0xffffffffu, q, 1);
                rstd = rsqrtf(q / (float)p.ln_c + 1e-5f);
            }
#pragma unroll
            for (int i = 0; i < NV; i += 2) {
                float4 f0 = *reinterpret_cast<const float4 *>(&areg[i]), f1 = *reinterpret_cast<const float4 *>(&areg[i + 1]);
                if (LN) {       // gamma / beta are zero on the padded channels: they stay exactly zero
                    const float *g = ln_s + lh * CPT + 4 * i, *be = ln_s + KP + lh * CPT + 4 * i;
                    f0.x = (f0.x - mean) * rstd * g[0] + be[0]; f0.y = (f0.y - mean) * rstd * g[1] + be[1];
                    f0.z = (f0.z - mean) * rstd * g[2] + be[2]; f0.w = (f0.w - mean) * rstd * g[3] + be[3];
                    f1.x = (f1.x - mean) * rstd * g[4] + be[4]; f1.y = (f1.y - mean) * rstd * g[5] + be[5];
                    f1.z = (f1.z - mean) * rstd * g[6] + be[6]; f1.w = (f1.w - mean) * rstd * g[7] + be[7];
                }
                *reinterpret_cast<uint4 *>(d + (i / 2) * A_LBO) =
                    make_uint4(pack_bf16(f0.x, f0.y), pack_bf16(f0.z, f0.w), pack_bf16(f1.x, f1.y), pack_bf16(f1.z, f1.w));
            }
        }
    };
    constexpr uint32_t IDESC = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
    auto issue = [&](int i, uint32_t tmem_d) {       // one thread: the KP/16 MMAs of tile i
        tc_fence_after();
        const uint32_t a0 = smem_u32(As + (i & 1) * A_STAGE), b0 = smem_u32(Bs);
#pragma unroll
        for (int j = 0; j < KP / 16; ++j)
            mma_f16(tmem_d + (uint32_t)((i & 1) * BUF1), make_desc(a0 + 2 * j * A_LBO, A_LBO, 128), make_desc(b0 + 2 * j * B_LBO, B_LBO, 128),
                    IDESC, j > 0 ? 1u : 0u);
        mma_commit(&mbar[i & 1]);
    };

    // residual rows of the tile about to be finished, fetched before the CTA turns to the next tile's
    // operands so that their latency hides behind a_store / the barrier / the MMA wait
    constexpr bool PRE = ((EPI & (EPI_RES1 | EPI_RES2)) != 0) && BN <= 64;
    constexpr int NR1 = (PRE && (EPI & EPI_RES1)) ? BN / 8 : 1, NR2 = (PRE && (EPI & EPI_RES2)) ? BN / 16 : 1;
    uint4 rreg1[NR1], rreg2[NR2];
    auto r_fetch = [&](int tile) {
        if (!PRE) return;
        const int m = tile * BM + 32 * (warp & 3) + lane;
        if (m >= p.rows) return;
        const long long row = (long long)b * p.rows + m;
        const int n0 = n_base + (warp >> 2) * (BN / 2);
        if (EPI & EPI_RES1) {
#pragma unroll
            for (int i = 0; i < NR1; ++i) rreg1[i] = *(reinterpret_cast<const uint4 *>(p.res1 + row * p.ldr1 + n0) + i);
        }
        if (EPI & EPI_RES2) {
#pragma unroll
            for (int i = 0; i < NR2; ++i) rreg2[i] = *(reinterpret_cast<const uint4 *>(p.res2 + row * p.ldr2 + n0) + i);
        }
    };

    if (n_my > 0) a_fetch(blockIdx.x);
    if (LN) __syncthreads();                 // gamma / beta are read from shared memory by a_store
    if (n_my > 0) a_store(0);
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_d = tmem_base_s;
    if (n_my > 0 && tid == 0) issue(0, tmem_d);
    if (n_my > 1) a_fetch(blockIdx.x + gridDim.x);
    for (int i = 0; i < n_my; ++i) {
        r_fetch(blockIdx.x + i * gridDim.x);
        if (i + 1 < n_my) {
            // stage (i+1)&1 was last read by the MMAs of tile i-1 and TMEM buffer (i+1)&1 drained by the
            // epilogue of tile i-1: both finished before this point in every thread's program order
            a_store((i + 1) & 1);
            fence_async_smem();
            tc_fence_before();
            __syncthreads();
            if (tid == 0) issue(i + 1, tmem_d);
            if (i + 2 < n_my) a_fetch(blockIdx.x + (i + 2) * gridDim.x);
        }
        mbar_wait(&mbar[i & 1], (uint32_t)((i >> 1) & 1));
        tc_fence_after();
        epilogue_tile<BN, EPI, PRE>(p, tmem_d + (uint32_t)((i & 1) * BUF1), b, (blockIdx.x + i * gridDim.x) * BM, n_base, warp, lane, rreg1, rreg2);
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_d), "n"(TMEM_COLS) : "memory");
    }
}

// ------------------------------------------------------------------------------------ TMA-fed pointwise GEMM
// The layers whose A operand already is bf16 (attention projection on v, FFN out on the hidden
// activations) are fed by the TMA engine: a 3-D tensor map {8 channels, rows, K/8} over the row-major
// activation matrix makes ONE cp.async.bulk.tensor per 128-row tile land in shared memory exactly in the
// canonical K-major UMMA layout (k-chunks of 8 channels, 128 rows of 16 bytes each) -- no thread loads,
// no register staging, no shared-memory stores, no proxy fence.  A ring of NS stages keeps NS tiles in
// flight; one thread waits on the stage's mbarrier and issues the tcgen05.mma of tile i+1 into the other
// TMEM buffer while all threads run the epilogue of tile i (residual rows prefetched one tile ahead).
template <int BN, int KP, int EPI>
__global__ void __launch_bounds__(GEMM_THREADS) gemm_tma_kernel(const __grid_constant__ GemmP p, const __grid_constant__ CUtensorMap tmA) {
    pdl_wait();
    constexpr int A_LBO = (BM / 8) * 128, B_LBO = (BN / 8) * 128;
    constexpr int A_STAGE = (KP / 8) * A_LBO;
    constexpr int NS = KP <= 64 ? 4 : 3;
    constexpr int TMEM_COLS = 2 * BN <= 32 ? 32 : (2 * BN <= 64 ? 64 : (2 * BN <= 128 ? 128 : (2 * BN <= 256 ? 256 : 512)));
    constexpr int BUF1 = TMEM_COLS / 2;
    extern __shared__ __align__(1024) uint8_t dsm[];
    uint8_t *As = dsm;                                        // [NS][A_STAGE]
    uint8_t *Bs = dsm + NS * A_STAGE;                         // [B_BYTES]
    __shared__ __align__(8) uint64_t full_bar[NS];
    __shared__ __align__(8) uint64_t mma_bar[2];
    __shared__ uint32_t tmem_base_s;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int b = blockIdx.z, n_base = blockIdx.y * BN;
    const int m_tiles = (p.rows + BM - 1) / BM;
    const int n_my = ((int)blockIdx.x < m_tiles) ? (m_tiles - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;

    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_s)), "n"(TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    if (tid == 32) {
#pragma unroll
        for (int s = 0; s < NS; ++s) mbar_init(&full_bar[s], 1);
        mbar_init(&mma_bar[0], 1);
        mbar_init(&mma_bar[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    {   // resident weight tile
        const bf16 *Wb = p.W + (long long)b * p.w_bstride;
        constexpr int NVEC = BN * (KP / 8), BATCH = 8;
        for (int i0 = 0; i0 < NVEC; i0 += BATCH * GEMM_THREADS) {
            uint4 wv[BATCH];
#pragma unroll
            for (int u = 0; u < BATCH; ++u) {
                const int idx = i0 + u * GEMM_THREADS + tid;
                if (idx < NVEC) {
                    const int n = idx / (KP / 8), q = idx - n * (KP / 8);
                    wv[u] = __ldg(reinterpret_cast<const uint4 *>(Wb + (long long)(n_base + n) * p.K) + q);
                }
            }
#pragma unroll
            for (int u = 0; u < BATCH; ++u) {
                const int idx = i0 + u * GEMM_THREADS + tid;
                if (idx < NVEC) {
                    const int n = idx / (KP / 8), q = idx - n * (KP / 8);
                    *reinterpret_cast<uint4 *>(Bs + q * B_LBO + (n >> 3) * 128 + (n & 7) * 16) = wv[u];
                }
            }
        }
    }
    constexpr bool PRE = ((EPI & (EPI_RES1 | EPI_RES2)) != 0) && BN <= 64;
    constexpr int NR1 = (PRE && (EPI & EPI_RES1)) ? BN / 8 : 1, NR2 = (PRE && (EPI & EPI_RES2)) ? BN / 16 : 1;
    uint4 rreg1[NR1], rreg2[NR2];
    auto r_fetch = [&](int tile) {
        if (!PRE) return;
        const int m = tile * BM + 32 * (warp & 3) + lane;
        if (m >= p.rows) return;
        const long long row = (long long)b * p.rows + m;
        const int n0 = n_base + (warp >> 2) * (BN / 2);
        if (EPI & EPI_RES1) {
#pragma unroll
            for (int i = 0; i < NR1; ++i) rreg1[i] = *(reinterpret_cast<const uint4 *>(p.res1 + row * p.ldr1 + n0) + i);
        }
        if (EPI & EPI_RES2) {
#pragma unroll
            for (int i = 0; i < NR2; ++i) rreg2[i] = *(reinterpret_cast<const uint4 *>(p.res2 + row * p.ldr2 + n0) + i);
        }
    };
    auto tma_load = [&](int i) {                              // one thread: tile i of this CTA -> stage i % NS
        const int st = i % NS;
        const int row0 = b * p.rows + (blockIdx.x + i * gridDim.x) * BM;
        const uint32_t bar = smem_u32(&full_bar[st]);
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"((uint32_t)A_STAGE) : "memory");
        asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
                     ::"r"(smem_u32(As + st * A_STAGE)), "l"(&tmA), "r"(0), "r"(row0), "r"(0), "r"(bar) : "memory");
    };
    constexpr uint32_t IDESC = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
    auto issue = [&](int i, uint32_t tmem_d) {                // one thread: wait for the stage, KP/16 MMAs
        mbar_wait(&full_bar[i % NS], (uint32_t)((i / NS) & 1));
        tc_fence_after();
        const uint32_t a0 = smem_u32(As + (i % NS) * A_STAGE), b0 = smem_u32(Bs);
#pragma unroll
        for (int j = 0; j < KP / 16; ++j)
            mma_f16(tmem_d + (uint32_t)((i & 1) * BUF1), make_desc(a0 + 2 * j * A_LBO, A_LBO, 128), make_desc(b0 + 2 * j * B_LBO, B_LBO, 128),
                    IDESC, j > 0 ? 1u : 0u);
        mma_commit(&mma_bar[i & 1]);
    };

    fence_async_smem();                                       // weight tile (generic stores) -> tensor core (async proxy)
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_d = tmem_base_s;
    if (tid == 0) {
        for (int i = 0; i < NS && i < n_my; ++i) tma_load(i);
        if (n_my > 0) issue(0, tmem_d);
    }
    for (int i = 0; i < n_my; ++i) {
        r_fetch(blockIdx.x + i * gridDim.x);
        if (tid == 0 && i + 1 < n_my) issue(i + 1, tmem_d);    // TMEM buffer (i+1)&1 was drained before the barrier below
        mbar_wait(&mma_bar[i & 1], (uint32_t)((i >> 1) & 1));
        tc_fence_after();
        if (tid == 0 && i + NS < n_my) tma_load(i + NS);       // stage i % NS: its MMAs have completed
        epilogue_tile<BN, EPI, PRE>(p, tmem_d + (uint32_t)((i & 1) * BUF1), b, (blockIdx.x + i * gridDim.x) * BM, n_base, warp, lane, rreg1, rreg2);
        tc_fence_before();
        __syncthreads();
    }
    if (warp == 0) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_d), "n"(TMEM_COLS) : "memory");
    }
}

// The same pipeline for a layer whose A operand is the fp32 residual stream (q | k | v): the tensor map is
// over fp32 rows {4 channels, rows, K/4} and the contraction runs as tcgen05.mma kind::tf32 (the tensor
// core reads the fp32 bits, 10 mantissa bits -- no less than the bf16 operands of the other layers), so
// the activations go HBM -> TMA -> shared memory -> tensor core without passing through a thread.
template <int BN, int KP, int EPI>
__global__ void __launch_bounds__(GEMM_THREADS) gemm_tma32_kernel(const __grid_constant__ GemmP p, const __grid_constant__ CUtensorMap tmA) {
    pdl_wait();
    constexpr int A_LBO = (BM / 8) * 128, B_LBO = (BN / 8) * 128;
    constexpr int A_STAGE = (KP / 4) * A_LBO;               // fp32 operands: k-chunks of 4 elements (16 bytes)
    constexpr int NS = KP <= 32 ? 4 : (KP <= 64 ? 3 : 2);
    constexpr int TMEM_COLS = 2 * BN <= 32 ? 32 : (2 * BN <= 64 ? 64 : (2 * BN <= 128 ? 128 : (2 * BN <= 256 ? 256 : 512)));
    constexpr int BUF1 = TMEM_COLS / 2;
    extern __shared__ __align__(1024) uint8_t dsm[];
    uint8_t *As = dsm;                                        // [NS][A_STAGE]
    uint8_t *Bs = dsm + NS * A_STAGE;                         // [B_BYTES]
    __shared__ __align__(8) uint64_t full_bar[NS];
    __shared__ __align__(8) uint64_t mma_bar[2];
    __shared__ uint32_t tmem_base_s;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int b = blockIdx.z, n_base = blockIdx.y * BN;
    const int m_tiles = (p.rows + BM - 1) / BM;
    const int n_my = ((int)blockIdx.x < m_tiles) ? (m_tiles - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;

    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_s)), "n"(TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    if (tid == 32) {
#pragma unroll
        for (int s = 0; s < NS; ++s) mbar_init(&full_bar[s], 1);
        mbar_init(&mma_bar[0], 1);
        mbar_init(&mma_bar[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (p.zero_ptr && blockIdx.x == 0 && blockIdx.y == 0 && blockIdx.z == 0)
        for (int i = tid; i < p.zero_n; i += GEMM_THREADS) p.zero_ptr[i] = 0.f;
    {   // resident weight tile (fp32 / tf32)
        const float *Wb = p.W32;
        constexpr int NVEC = BN * (KP / 4), BATCH = 8;
        for (int i0 = 0; i0 < NVEC; i0 += BATCH * GEMM_THREADS) {
            uint4 wv[BATCH];
#pragma unroll
            for (int u = 0; u < BATCH; ++u) {
                const int idx = i0 + u * GEMM_THREADS + tid;
                if (idx < NVEC) {
                    const int n = idx / (KP / 4), q = idx - n * (KP / 4);
                    wv[u] = __ldg(reinterpret_cast<const uint4 *>(Wb + (long long)(n_base + n) * p.K) + q);
                }
            }
#pragma unroll
            for (int u = 0; u < BATCH; ++u) {
                const int idx = i0 + u * GEMM_THREADS + tid;
                if (idx < NVEC) {
                    const int n = idx / (KP / 4), q = idx - n * (KP / 4);
                    *reinterpret_cast<uint4 *>(Bs + q * B_LBO + (n >> 3) * 128 + (n & 7) * 16) = wv[u];
                }
            }
        }
    }
    constexpr bool PRE = ((EPI & (EPI_RES1 | EPI_RES2)) != 0) && BN <= 64;
    constexpr int NR1 = (PRE && (EPI & EPI_RES1)) ? BN / 8 : 1, NR2 = (PRE && (EPI & EPI_RES2)) ? BN / 16 : 1;
    uint4 rreg1[NR1], rreg2[NR2];
    auto r_fetch = [&](int tile) {
        if (!PRE) return;
        const int m = tile * BM + 32 * (warp & 3) + lane;
        if (m >= p.rows) return;
        const long long row = (long long)b * p.rows + m;
        const int n0 = n_base + (warp >> 2) * (BN / 2);
        if (EPI & EPI_RES1) {
#pragma unroll
            for (int i = 0; i < NR1; ++i) rreg1[i] = *(reinterpret_cast<const uint4 *>(p.res1 + row * p.ldr1 + n0) + i);
        }
        if (EPI & EPI_RES2) {
#pragma unroll
            for (int i = 0; i < NR2; ++i) rreg2[i] = *(reinterpret_cast<const uint4 *>(p.res2 + row * p.ldr2 + n0) + i);
        }
    };
    auto tma_load = [&](int i) {                              // one thread: tile i of this CTA -> stage i % NS
        const int st = i % NS;
        const int row0 = b * p.rows + (blockIdx.x + i * gridDim.x) * BM;
        const uint32_t bar = smem_u32(&full_bar[st]);
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"((uint32_t)A_STAGE) : "memory");
        asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
                     ::"r"(smem_u32(As + st * A_STAGE)), "l"(&tmA), "r"(0), "r"(row0), "r"(0), "r"(bar) : "memory");
    };
    // instruction descriptor: D = F32, A = B = TF32 (format 2), both K-major
    constexpr uint32_t IDESC = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
    auto issue = [&](int i, uint32_t tmem_d) {                // one thread: wait for the stage, KP/8 MMAs (K = 8 each)
        mbar_wait(&full_bar[i % NS], (uint32_t)((i / NS) & 1));
        tc_fence_after();
        const uint32_t a0 = smem_u32(As + (i % NS) * A_STAGE), b0 = smem_u32(Bs);
#pragma unroll
        for (int j = 0; j < KP / 8; ++j)
            mma_tf32(tmem_d + (uint32_t)((i & 1) * BUF1), make_desc(a0 + 2 * j * A_LBO, A_LBO, 128), make_desc(b0 + 2 * j * B_LBO, B_LBO, 128),
                    IDESC, j > 0 ? 1u : 0u);
        mma_commit(&mma_bar[i & 1]);
    };

    fence_async_smem();                                       // weight tile (generic stores) -> tensor core (async proxy)
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_d = tmem_base_s;
    if (tid == 0) {
        for (int i = 0; i < NS && i < n_my; ++i) tma_load(i);
        if (n_my > 0) issue(0, tmem_d);
    }
    for (int i = 0; i < n_my; ++i) {
        r_fetch(blockIdx.x + i * gridDim.x);
        if (tid == 0 && i + 1 < n_my) issue(i + 1, tmem_d);    // TMEM buffer (i+1)&1 was drained before the barrier below
        mbar_wait(&mma_bar[i & 1], (uint32_t)((i >> 1) & 1));
        tc_fence_after();
        if (tid == 0 && i + NS < n_my) tma_load(i + NS);       // stage i % NS: its MMAs have completed
        epilogue_tile<BN, EPI, PRE>(p, tmem_d + (uint32_t)((i & 1) * BUF1), b, (blockIdx.x + i * gridDim.x) * BM, n_base, warp, lane, rreg1, rreg2);
        tc_fence_before();
        __syncthreads();
    }
    if (warp == 0) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_d), "n"(TMEM_COLS) : "memory");
    }
}

// ------------------------------------------------------------------------------------ row-streaming 3x3 convolution
// Conv2d(32, 32, 3, padding 1) on the full-resolution level (embedding / mapping convs of every MST
// body and conv_out).  The K-chunked kernel above gathers every input pixel nine times through L2
// (288 MB per launch, ~3.6 TB/s: 75-90 us).  Here a CTA owns a strip of 128 columns and walks down a
// segment of rows; each input row enters shared memory ONCE (fp32 -> bf16, canonical K-major rows of
// 16 bytes, 130 pixels incl. the x halo, zeros outside the map) into a ring of four row slots, and an
// output row is 9 taps x 2 tcgen05.mma (M = 128 pixels, N = 32, K = 16) whose A descriptors simply
// start (dx * 16 B) into the slot of row y + dy - 1 -- the canonical layout is linear in the pixel
// index, so a shifted window is a shifted start address.  Software pipeline per output row:
//   store row y+1 (registers -> slot), barrier, issue the 18 MMAs of row y into TMEM buffer y&1,
//   fetch row y+2 (registers), wait for row y-1, epilogue of row y-1 (residual, store / crop).
constexpr int C3_PXP = 138;                       // pixels per slot row (130 used); 138 staggers the four k-chunks over the banks
constexpr int C3_LBO = C3_PXP * 16;               // bytes between k-chunks of 8 channels
constexpr int C3_SLOT = 4 * C3_LBO;               // 32 channels
constexpr int C3_SLOTS = 4;
constexpr int C3_B_LBO = (32 / 8) * 128;          // weights: 32 output channels per k-chunk
constexpr int C3_SMEM = C3_SLOTS * C3_SLOT + 36 * C3_B_LBO;

template <int EPI>
__global__ void __launch_bounds__(GEMM_THREADS) conv3_stream_kernel(const __grid_constant__ GemmP p, int seg_rows) {
    pdl_wait();
    extern __shared__ __align__(1024) uint8_t dsm[];
    uint8_t *ring = dsm;                                   // [C3_SLOTS][4 k-chunks][C3_PXP][16 B]
    uint8_t *Bs = dsm + C3_SLOTS * C3_SLOT;                // [36 k-chunks][32 n][16 B]
    __shared__ __align__(8) uint64_t mbar[2];
    __shared__ uint32_t tmem_base_s;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int b = blockIdx.z, x0 = blockIdx.x * BM;
    const int H = p.Hi, W = p.Wi;
    const int y_begin = blockIdx.y * seg_rows, y_end = min(H, y_begin + seg_rows);
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_s)), "n"(64) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    if (tid == 32) {
        mbar_init(&mbar[0], 1);
        mbar_init(&mbar[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    // resident weights: [32][288] bf16 -> canonical K-major
    for (int idx = tid; idx < 32 * 36; idx += GEMM_THREADS) {
        const int n = idx / 36, q = idx - n * 36;
        *reinterpret_cast<uint4 *>(Bs + q * C3_B_LBO + (n >> 3) * 128 + (n & 7) * 16) =
            __ldg(reinterpret_cast<const uint4 *>(p.W + (long long)n * 288) + q);
    }
    // ---- row loader: 130 pixels x 32 fp32 channels = 1040 float4 quads -> 5 per thread (last partial)
    constexpr int QPT = (130 * 8 + GEMM_THREADS - 1) / GEMM_THREADS;       // 5
    float4 rreg[QPT];
    const float *A = reinterpret_cast<const float *>(p.A1) + (long long)b * H * W * 32;
    auto fetch = [&](int y) {
#pragma unroll
        for (int u = 0; u < QPT; ++u) {
            const int idx = tid + u * GEMM_THREADS;         // quad index: pixel idx / 8, channels 4*(idx % 8) ..
            const int px = idx >> 3, xx = x0 - 1 + px;
            const bool ok = idx < 130 * 8 && (unsigned)y < (unsigned)H && (unsigned)xx < (unsigned)W;
            rreg[u] = ok ? __ldg(reinterpret_cast<const float4 *>(A + ((long long)y * W + xx) * 32) + (idx & 7)) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
    };
    auto store = [&](int y) {                              // row y -> slot y & 3 (y may be -1: slot 3)
        uint8_t *slot = ring + ((y + 4) & 3) * C3_SLOT;
#pragma unroll
        for (int u = 0; u < QPT; ++u) {
            const int idx = tid + u * GEMM_THREADS;
            if (idx < 130 * 8) {
                const int px = idx >> 3, q = idx & 7;      // channels 4q .. 4q+3: k-chunk q/2, bytes 8*(q&1) ..
                *reinterpret_cast<uint2 *>(slot + (q >> 1) * C3_LBO + px * 16 + (q & 1) * 8) =
                    make_uint2(pack_bf16(rreg[u].x, rreg[u].y), pack_bf16(rreg[u].z, rreg[u].w));
            }
        }
    };
    constexpr uint32_t IDESC = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(32 >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
    auto issue = [&](int y, uint32_t tmem_d) {             // one thread: 9 taps x 2 MMAs of output row y
        tc_fence_after();
        const uint32_t r0 = smem_u32(ring), b0 = smem_u32(Bs);
#pragma unroll
        for (int t = 0; t < 9; ++t) {
            const int dy = t / 3, dx = t % 3;
            const uint32_t a0 = r0 + (uint32_t)(((y + dy - 1 + 4) & 3) * C3_SLOT) + (uint32_t)(dx * 16);
#pragma unroll
            for (int j = 0; j < 2; ++j)
                mma_f16(tmem_d + (uint32_t)((y & 1) * 32), make_desc(a0 + 2 * j * C3_LBO, C3_LBO, 128),
                        make_desc(b0 + (4 * t + 2 * j) * C3_B_LBO, C3_B_LBO, 128), IDESC, (t > 0 || j > 0) ? 1u : 0u);
        }
        mma_commit(&mbar[y & 1]);
    };

    fetch(y_begin - 1);
    store(y_begin - 1);
    fetch(y_begin);
    store(y_begin);
    fetch(y_begin + 1);
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_d = tmem_base_s;
    uint32_t ph[2] = {0u, 0u};
    for (int y = y_begin; y < y_end; ++y) {
        // slot (y+1)&3 last held row y-3, read by the MMAs of row y-2 whose completion was awaited in
        // iteration y-1; TMEM buffer y&1 was drained by the epilogue of row y-2 (iteration y-1)
        store(y + 1);
        fence_async_smem();
        tc_fence_before();
        __syncthreads();
        if (tid == 0) issue(y, tmem_d);
        if (y + 1 < y_end) fetch(y + 2);
        if (y > y_begin) {
            const int yp = y - 1;
            mbar_wait(&mbar[yp & 1], ph[yp & 1]);
            ph[yp & 1] ^= 1u;
            tc_fence_after();
            epilogue_tile<32, EPI>(p, tmem_d + (uint32_t)((yp & 1) * 32), b, yp * W + x0, 0, warp, lane);
        }
    }
    {
        const int yp = y_end - 1;
        mbar_wait(&mbar[yp & 1], ph[yp & 1]);
        tc_fence_after();
        epilogue_tile<32, EPI>(p, tmem_d + (uint32_t)((yp & 1) * 32), b, yp * W + x0, 0, warp, lane);
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_d), "n"(64) : "memory");
    }
}

// ------------------------------------------------------------------------------------ fused feed-forward block
// FeedForward of an MSAB (MST_Plus_Plus.py:141-158 behind the PreNorm of :57-65)
//     x += W4 . GELU( dw3x3( GELU( W0 . LayerNorm(x) ) ) )
// in ONE kernel per 128 hidden channels: the 4c-wide hidden maps never reach HBM (the three-kernel form wrote and read
// 2 x 256 B per pixel of them at the full-resolution level).  A CTA owns a strip of <= 126 columns and walks down a
// segment of rows; per image row (M = 128 pixels = strip + x halo):
//   in :  T1[128 px][128 hidden] = LN(x row)[128][CP] . W0^T        CP/16 tcgen05.mma, N = 128, accumulator in TMEM
//   E1 :  T1 -> f16 -> GELU (packed f16) -> ring slot of the row ([px][128 ch], zeros outside the map = the conv's padding)
//   dw :  depthwise 3x3 on the CUDA cores from three ring rows: lane = 4 channels (its 9 x 4 taps live in registers as
//         half2), warp = a run of 8 pixels, packed HFMA2 (f16 keeps 11 mantissa bits through the nine-term sum: less
//         rounding than ONE bf16 store of the three-kernel form), -> GELU (packed f16) -> f16 A operand of the out GEMM
//   out:  T3[128 px][CP] = hidden2[128][128] . W4^T                 8 tcgen05.mma, N = CP
//   E3 :  T3 + residual row -> x
// Warp-specialised: 16 loader / epilogue warps run  E1(h), stage LN(x row h+1) | E3(h-2), dw(h-1)  per hidden row h, a 17th
// warp issues  in(h+1) | out(h-1);  hand-offs are mbarriers (tcgen05.commit one way, one arrival per warp the other) plus
// ONE named barrier per row among the 16 warps (row h of the ring complete); the ring has four slots so that the write of
// row h+1 never meets a reader of row h-3.  Measured dead end: the depthwise conv as 72 tcgen05.mma per row (N = 16,
// diagonal 16x16 tap tiles, A descriptors shifted by dx * 16 B): correct, but an M = 128 MMA re-reads its 4 KB A tile from
// shared memory in ~128 clk whatever N is -- 144 us per launch against 153 us for the three kernels it replaced.
// It serves the full-resolution level (Cp = 32, 124 hidden channels: one pass); the coarser levels measured faster as three
// kernels.  Wider hidden maps run as one pass per 128-channel chunk: chunk 0 writes x = xin + part0, chunk c adds
// part_c in place (stream order: the sum order is fixed, the forward stays bit-reproducible); LN(xin) is recomputed.
struct FfnP {
    const float *xin;          // [B, H, W, CP] fp32: the residual stream after the attention block (LayerNorm input)
    const float *res;          // rows the chunk's contribution is added to (xin for chunk 0, out afterwards)
    float *out;                // [B, H, W, CP]; never aliases xin (halo rows of xin are read while neighbours write out)
    const uint8_t *wblob;      // this chunk's GEMM operands in shared-memory layout: W0 | W4
    const float *dw_w;         // depthwise taps of this chunk: [9][dw_stride] fp32, 128 channels used
    const float *ln_g, *ln_b;
    int dw_stride, ln_c, H, W, strip_w, seg_rows;
};
constexpr int FF_HC = 128;                                  // hidden channels per pass
constexpr int FF_PXS = 2 * FF_HC + 16;                      // ring bytes per pixel: 128 f16 channels + 16 (conflict-free row-per-lane stores)
constexpr int FF_SLOT = 128 * FF_PXS;
constexpr int FF_SLOTS = 4;
constexpr int FF_ALBO = 2048 + 16;                          // out-GEMM A operand: bytes between k-chunks (padded: conflict-free 8-byte stores)
constexpr int FF_AOUT = (FF_HC / 8) * FF_ALBO;
constexpr int FF_TMEM_T1 = 0, FF_TMEM_T3 = 128;
template <int CP>
struct FfnCfg {
    static constexpr int W0_BYTES = (CP / 8) * 2048;        // [CP/8 k-chunks][128 n][16 B]
    static constexpr int W4_BYTES = (FF_HC / 8) * CP * 16;  // [16 k-chunks][CP n][16 B]
    static constexpr int BLOB = W0_BYTES + W4_BYTES;
    static constexpr int AIN = (CP / 8) * 2048;
    static constexpr int SMEM = FF_SLOTS * FF_SLOT + FF_AOUT + AIN + BLOB + 2 * CP * 4;
};
constexpr int FF_EPI_WARPS = 16;                            // loader / epilogue warps; one more warp issues the MMAs
constexpr int FF_THREADS = (FF_EPI_WARPS + 1) * 32;

template <int N>
__device__ __forceinline__ void tmem_ldn(uint32_t taddr, float (&v)[N]) {
    static_assert(N == 8 || N == 16 || N == 32, "tcgen05.ld shapes used here");
    uint32_t r[N];
    if constexpr (N == 8) {
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                     : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]) : "r"(taddr));
    } else if constexpr (N == 16) {
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                     : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                       "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
                     : "r"(taddr));
    } else {
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
                     "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
                     : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                       "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
                       "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
                       "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
                     : "r"(taddr));
    }
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < N; ++i) v[i] = __uint_as_float(r[i]);
}

// GELU of the packed-f16 stages (both hidden-map stages of the fused feed-forward kernel, the positional embedding, the
// coarse-level depthwise conv; the fused kernel alone evaluates 256 per pixel and the SFU is their bound):
//   x Phi(x) = x/2 (1 + tanh(x (a1 + a3 x^2))),  minimax fit of the cubic argument polynomial: |error| < 2.7e-4 absolute before the
// 2^-11 relative error of tanh.approx, an order of magnitude inside the bf16 rounding of the maps it produces; monotonic for every
// x, so overflowing inputs saturate to x / 0 instead of turning over (a quintic fit is ten times closer but bends back beyond
// |x| = 11); 9 instructions per PAIR of values including the two SFU operations (the erfc form of gelu() takes 14 per value).
__device__ __forceinline__ __half2 gelu_h2(__half2 x) {
    const __half2 a1 = __float2half2_rn(0.8001570785f), a3 = __float2half2_rn(0.0347008934f), hf = __float2half2_rn(0.5f);
    const __half2 t = __hmul2(__hfma2(__hmul2(x, x), a3, a1), x);
    uint32_t th;
    asm("tanh.approx.f16x2 %0, %1;" : "=r"(th) : "r"(*reinterpret_cast<const uint32_t *>(&t)));
    const __half2 hx = __hmul2(x, hf);
    return __hfma2(hx, *reinterpret_cast<const __half2 *>(&th), hx);
}
__device__ __forceinline__ __half2 f2h2_sat(float lo, float hi) {       // round to f16, clamped to the finite range
    uint32_t r;
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    return *reinterpret_cast<const __half2 *>(&r);
}
// tcgen05.ld of 32 columns split into issue and wait, so that independent work can sit between the two; the wait names
// the registers as read-write operands: nothing that uses them can be scheduled above it
__device__ __forceinline__ void tmem_ld32_issue(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
                 "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                   "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
                   "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
                   "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
                 : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld32_wait(uint32_t (&r)[32]) {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]),
                   "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15]),
                   "+r"(r[16]), "+r"(r[17]), "+r"(r[18]), "+r"(r[19]), "+r"(r[20]), "+r"(r[21]), "+r"(r[22]), "+r"(r[23]),
                   "+r"(r[24]), "+r"(r[25]), "+r"(r[26]), "+r"(r[27]), "+r"(r[28]), "+r"(r[29]), "+r"(r[30]), "+r"(r[31])
                 :: "memory");
}

__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// UMMA descriptor from its two 32-bit halves (the low word holds the start address >> 4 and the LBO, so stepping through
// operand tiles is one integer add on it)
__device__ __forceinline__ void mma_f16_lh(uint32_t tmem_d, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi, uint32_t idesc,
                                           uint32_t accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\tmov.b64 da, {%1, %2};\n\tmov.b64 db, {%3, %4};\n\tsetp.ne.b32 p, %6, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, p;\n\t}"
                 ::"r"(tmem_d), "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ uint32_t desc_lo(uint32_t saddr, uint32_t lbo_bytes) { return ((saddr & 0x3ffffu) >> 4) | ((lbo_bytes >> 4) << 16); }
constexpr uint32_t DESC_HI_SBO128 = (128u >> 4) | (1u << 14);       // SBO = 128 B, descriptor version 1, no swizzle

template <int CP>
__global__ void __launch_bounds__(FF_THREADS, 1) ffn_fused_kernel(const __grid_constant__ FfnP p) {
    typedef FfnCfg<CP> Cfg;
    extern __shared__ __align__(1024) uint8_t dsm[];
    uint8_t *ring = dsm;                                    // [4 slots][128 px][272 B]: f16 hidden rows
    uint8_t *Aout = ring + FF_SLOTS * FF_SLOT;              // [16 k-chunks][128 px][16 B], k-chunks FF_ALBO apart
    uint8_t *Ain = Aout + FF_AOUT;                          // [CP/8 k-chunks][128 px][16 B]
    uint8_t *W0s = Ain + Cfg::AIN;
    uint8_t *W4s = W0s + Cfg::W0_BYTES;
    float *ln_s = reinterpret_cast<float *>(W0s + Cfg::BLOB);            // gamma[CP] | beta[CP]
    // 0: weights landed; 1: in, 2: out (tcgen05.commit); 3: E1 done + next LN row staged, 4: dw row staged (one arrival per warp)
    __shared__ __align__(8) uint64_t bars[5];
    __shared__ uint32_t tmem_base_s;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int b = blockIdx.z, H = p.H, W = p.W;
    const int xs = blockIdx.x * p.strip_w;                  // first output column of the strip
    const int wv = min(p.strip_w, W - xs);                  // output columns of this strip
    const int y_begin = blockIdx.y * p.seg_rows, y_end = min(H, y_begin + p.seg_rows);
    const int h0 = y_begin - 1;

    // ---- set-up that does not depend on the preceding kernel (overlaps its tail under programmatic dependent launch): barriers,
    // the weight copy, LayerNorm parameters.  NOT the TMEM allocation: a CTA that holds tensor memory while it waits for its
    // predecessor can starve that predecessor's CTAs that are not resident yet (measured with the same idea in the GEMM kernels:
    // TMEM + weights staged before griddepcontrol.wait made the forward 7 % slower, 3.00 -> 3.22 ms).
    if (tid == 0) {
        mbar_init(&bars[0], 1);
        mbar_init(&bars[1], 1);
        mbar_init(&bars[2], 1);
        mbar_init(&bars[3], FF_EPI_WARPS);
        mbar_init(&bars[4], FF_EPI_WARPS);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        // the chunk's GEMM operands are stored in their shared-memory layout: one bulk copy by the TMA engine
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(&bars[0])), "r"((uint32_t)Cfg::BLOB) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                     ::"r"(smem_u32(W0s)), "l"(p.wblob), "r"((uint32_t)Cfg::BLOB), "r"(smem_u32(&bars[0])) : "memory");
    }
    for (int i = tid; i < CP; i += FF_THREADS) {
        ln_s[i] = i < p.ln_c ? __ldg(p.ln_g + i) : 0.f;
        ln_s[CP + i] = i < p.ln_c ? __ldg(p.ln_b + i) : 0.f;
    }
    // rows 126, 127 of the out-GEMM operand are never produced (their outputs are discarded): keep them finite
    for (int i = tid; i < (FF_HC / 8) * 2; i += FF_THREADS)
        *reinterpret_cast<uint4 *>(Aout + (i >> 1) * FF_ALBO + (126 + (i & 1)) * 16) = make_uint4(0u, 0u, 0u, 0u);
    pdl_wait();
    if (warp == FF_EPI_WARPS) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_s)), "n"(256) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_d = tmem_base_s;

    if (warp == FF_EPI_WARPS) {
        // ================================================================ MMA issuer (one lane; the warp stays converged)
        constexpr uint32_t IDESC0 = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(BM >> 4) << 24);
        // in: A = B = bf16; out: A = B = f16 (the hidden map after the depthwise stage stays f16, W4 is stored as f16)
        constexpr uint32_t IDESC_IN = IDESC0 | ((uint32_t)(FF_HC >> 3) << 17);
        constexpr uint32_t IDESC_OUT = (1u << 4) | ((uint32_t)(BM >> 4) << 24) | ((uint32_t)(CP >> 3) << 17);
        const uint32_t ain_lo = desc_lo(smem_u32(Ain), 2048), w0_lo = desc_lo(smem_u32(W0s), 2048);
        const uint32_t aout_lo = desc_lo(smem_u32(Aout), FF_ALBO), w4_lo = desc_lo(smem_u32(W4s), CP * 16);
        auto issue_in = [&]() {
#pragma unroll
            for (int j = 0; j < CP / 16; ++j)
                mma_f16_lh(tmem_d + FF_TMEM_T1, ain_lo + j * (2 * 2048 / 16), DESC_HI_SBO128, w0_lo + j * (2 * 2048 / 16), DESC_HI_SBO128, IDESC_IN,
                           j > 0 ? 1u : 0u);
            mma_commit(&bars[1]);
        };
        auto issue_out = [&]() {
#pragma unroll
            for (int j = 0; j < FF_HC / 16; ++j)
                mma_f16_lh(tmem_d + FF_TMEM_T3, aout_lo + j * (2 * FF_ALBO / 16), DESC_HI_SBO128, w4_lo + j * (2 * CP * 16 / 16), DESC_HI_SBO128, IDESC_OUT,
                           j > 0 ? 1u : 0u);
            mma_commit(&bars[2]);
        };
        uint32_t ph_e1 = 0u, ph_e2 = 0u;
        mbar_wait(&bars[0], 0u);                                  // weights
        mbar_wait(&bars[3], ph_e1);                               // first LayerNorm row staged
        ph_e1 ^= 1u;
        tc_fence_after();
        if (lane == 0) issue_in();
        __syncwarp();
        for (int h = h0; h <= y_end; ++h) {
            mbar_wait(&bars[3], ph_e1);                           // T1 drained by E1(h), LN row h+1 staged
            ph_e1 ^= 1u;
            tc_fence_after();
            if (lane == 0 && h + 1 <= y_end) issue_in();
            __syncwarp();
            if (h - 1 >= y_begin) {
                mbar_wait(&bars[4], ph_e2);                       // dw row h-1 staged, T3 drained by E3(h-2)
                ph_e2 ^= 1u;
                tc_fence_after();
                if (lane == 0) issue_out();
                __syncwarp();
            }
        }
    } else {
        // ================================================================ loader / epilogue warps
        // depthwise taps of this lane's four channels, as half2 pairs, for the whole kernel
        __half2 wreg[9][2];
#pragma unroll
        for (int t = 0; t < 9; ++t) {
            const float4 wv4 = __ldg(reinterpret_cast<const float4 *>(p.dw_w + (long long)t * p.dw_stride + 4 * lane));
            wreg[t][0] = __floats2half2_rn(wv4.x, wv4.y);
            wreg[t][1] = __floats2half2_rn(wv4.z, wv4.w);
        }
        // x row loader: four threads per pixel, LayerNorm over the ln_c real channels in registers
        constexpr int CPT = CP / 4, NV = CPT / 4;              // 8 or 16 channels per thread = 2 or 4 float4
        const float ln_inv_c = 1.0f / (float)p.ln_c, ln_pad = (float)(CP - p.ln_c);
        const int lr = tid >> 2, lq = tid & 3;
        const int lx = xs - 1 + lr;
        const bool lx_ok = (unsigned)lx < (unsigned)W;
        // running 32-bit element offsets (advanced by one image row per call: no 64-bit index arithmetic in the loop;
        // the host refuses maps of 2^31 elements or more)
        const uint32_t row_pitch = (uint32_t)(W * CP);
        uint32_t a_off = (uint32_t)((((long long)b * H + h0) * W + lx) * CP + lq * CPT);         // row of the next a_fetch (wraps for row -1: unused)
        int a_row = h0;
        uint4 areg[NV];
        auto a_fetch = [&]() {
            if (lx_ok && (unsigned)a_row < (unsigned)H) {
                const uint4 *q = reinterpret_cast<const uint4 *>(p.xin + a_off);
#pragma unroll
                for (int i = 0; i < NV; ++i) areg[i] = __ldg(q + i);
            } else {
#pragma unroll
                for (int i = 0; i < NV; ++i) areg[i] = make_uint4(0u, 0u, 0u, 0u);
            }
            a_off += row_pitch;
            ++a_row;
        };
        auto a_store = [&]() {
            uint8_t *d = Ain + (lq * (CPT / 8)) * 2048 + lr * 16;
            const int ch0 = lq * CPT;
            // the padded channels of the residual stream are exactly zero: they add nothing to the sum, and (0 - mean)^2
            // each to the squared deviations, which is taken out again in closed form -- no per-channel masks
            float s = 0.f;
#pragma unroll
            for (int i = 0; i < NV; ++i) {
                const float4 f = *reinterpret_cast<const float4 *>(&areg[i]);
                s += (f.x + f.y) + (f.z + f.w);
            }
            s += __shfl_xor_sync(0xffffffffu, s, 1);
            s += __shfl_xor_sync(0xffffffffu, s, 2);
            const float mean = s * ln_inv_c;
            float q = 0.f;
#pragma unroll
            for (int i = 0; i < NV; ++i) {
                const float4 f = *reinterpret_cast<const float4 *>(&areg[i]);
                const float d0 = f.x - mean, d1 = f.y - mean, d2 = f.z - mean, d3 = f.w - mean;
                q += d0 * d0 + d1 * d1 + d2 * d2 + d3 * d3;
            }
            q += __shfl_xor_sync(0xffffffffu, q, 1);
            q += __shfl_xor_sync(0xffffffffu, q, 2);
            q = fmaxf(fmaf(-ln_pad, mean * mean, q), 0.f);
            const float rstd = rsqrtf(fmaf(q, ln_inv_c, 1e-5f));
#pragma unroll
            for (int i = 0; i < NV; i += 2) {       // gamma / beta are zero on the padded channels: they stay exactly zero
                float4 f0 = *reinterpret_cast<const float4 *>(&areg[i]), f1 = *reinterpret_cast<const float4 *>(&areg[i + 1]);
                const float *g = ln_s + ch0 + 4 * i, *be = ln_s + CP + ch0 + 4 * i;
                f0.x = (f0.x - mean) * rstd * g[0] + be[0]; f0.y = (f0.y - mean) * rstd * g[1] + be[1];
                f0.z = (f0.z - mean) * rstd * g[2] + be[2]; f0.w = (f0.w - mean) * rstd * g[3] + be[3];
                f1.x = (f1.x - mean) * rstd * g[4] + be[4]; f1.y = (f1.y - mean) * rstd * g[5] + be[5];
                f1.z = (f1.z - mean) * rstd * g[6] + be[6]; f1.w = (f1.w - mean) * rstd * g[7] + be[7];
                *reinterpret_cast<uint4 *>(d + (i / 2) * 2048) =
                    make_uint4(pack_bf16(f0.x, f0.y), pack_bf16(f0.z, f0.w), pack_bf16(f1.x, f1.y), pack_bf16(f1.z, f1.w));
            }
        };

        // E1 / E3: thread = (pixel em = TMEM lane, quarter eq of the columns)
        const int em = 32 * (warp & 3) + lane;
        const uint32_t lane_bits = (uint32_t)(32 * (warp & 3)) << 16;
        const int eq = warp >> 2;
        auto h2u = [](uint32_t lo, uint32_t hi) {    // two accumulator columns -> f16 pair -> GELU
            const __half2 t = gelu_h2(f2h2_sat(__uint_as_float(lo), __uint_as_float(hi)));
            return *reinterpret_cast<const uint32_t *>(&t);
        };
        // hidden row h -> ring slot (h may be -1), after staging the LayerNorm of row h+1
        auto e1 = [&](int h, bool stage_next) {
            const int x = xs - 1 + em;
            const bool live = (unsigned)h < (unsigned)H && (unsigned)x < (unsigned)W;
            uint8_t *dst = ring + ((h + 4) & 3) * FF_SLOT + em * FF_PXS + eq * 64;
            if (stage_next) a_store();                          // registers hold row h+1; in(h) has finished with the stage
            uint32_t v[32];
            tmem_ld32_issue(tmem_d + FF_TMEM_T1 + lane_bits + (uint32_t)(32 * eq), v);
            tmem_ld32_wait(v);
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                uint4 o = make_uint4(0u, 0u, 0u, 0u);
                if (live) o = make_uint4(h2u(v[8 * k], v[8 * k + 1]), h2u(v[8 * k + 2], v[8 * k + 3]), h2u(v[8 * k + 4], v[8 * k + 5]), h2u(v[8 * k + 6], v[8 * k + 7]));
                *reinterpret_cast<uint4 *>(dst + 16 * k) = o;
            }
        };
        // the residual values E3(y) adds are fetched into registers one stage ahead of their use
        constexpr int QC = CP / 4;                              // 8 or 16 output channels per thread
        float4 rres[QC / 4];
        // residual / output rows advance with every res_fetch / e3 call (one per output row, in order)
        uint32_t r_off = (uint32_t)(((((long long)b * H + y_begin) * W) + xs + em) * CP + QC * eq), o_off = r_off;
        auto res_fetch = [&]() {
            if (em < wv) {
                const float4 *q = reinterpret_cast<const float4 *>(p.res + r_off);
#pragma unroll
                for (int i = 0; i < QC / 4; ++i) rres[i] = q[i];
            }
            r_off += row_pitch;
        };
        auto e3 = [&]() {
            float v[QC];
            tmem_ldn<QC>(tmem_d + FF_TMEM_T3 + lane_bits + (uint32_t)(QC * eq), v);
            if (em < wv) {
#pragma unroll
                for (int i = 0; i < QC; i += 4) {
                    const float4 r = rres[i / 4];
                    *reinterpret_cast<float4 *>(p.out + o_off + i) = make_float4(v[i] + r.x, v[i + 1] + r.y, v[i + 2] + r.z, v[i + 3] + r.w);
                }
            }
            o_off += row_pitch;
        };
        // depthwise 3x3 + GELU of output row y: warp = output pixels 8 warp .. 8 warp + 7 (ring pixel + 1 is the centre),
        // lane = channels 4 lane .. 4 lane + 3; two half-runs of four pixels from a 3 x 6 register window
        auto dw = [&](int y) {
            const uint8_t *r0 = ring + ((y + 3) & 3) * FF_SLOT + lane * 8;
            const uint8_t *r1 = ring + ((y + 4) & 3) * FF_SLOT + lane * 8;
            const uint8_t *r2 = ring + ((y + 5) & 3) * FF_SLOT + lane * 8;
            uint8_t *ao = Aout + (lane >> 1) * FF_ALBO + (lane & 1) * 8;
#pragma unroll
            for (int hf = 0; hf < 2; ++hf) {
                const int p0 = 8 * warp + 4 * hf;
                uint2 v[3][6];
#pragma unroll
                for (int c = 0; c < 6; ++c) {
                    const int px = min(p0 + c, 127);              // pixels 128, 129 only feed the discarded outputs 126, 127
                    v[0][c] = *reinterpret_cast<const uint2 *>(r0 + px * FF_PXS);
                    v[1][c] = *reinterpret_cast<const uint2 *>(r1 + px * FF_PXS);
                    v[2][c] = *reinterpret_cast<const uint2 *>(r2 + px * FF_PXS);
                }
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    __half2 a0 = __hmul2(*reinterpret_cast<const __half2 *>(&v[0][j].x), wreg[0][0]);
                    __half2 a1 = __hmul2(*reinterpret_cast<const __half2 *>(&v[0][j].y), wreg[0][1]);
#pragma unroll
                    for (int t = 1; t < 9; ++t) {
                        const uint2 &u = v[t / 3][j + t % 3];
                        a0 = __hfma2(*reinterpret_cast<const __half2 *>(&u.x), wreg[t][0], a0);
                        a1 = __hfma2(*reinterpret_cast<const __half2 *>(&u.y), wreg[t][1], a1);
                    }
                    a0 = gelu_h2(a0);
                    a1 = gelu_h2(a1);
                    const int m = p0 + j;
                    if (m < 126)
                        *reinterpret_cast<uint2 *>(ao + m * 16) = make_uint2(*reinterpret_cast<const uint32_t *>(&a0), *reinterpret_cast<const uint32_t *>(&a1));
                }
            }
        };
        auto publish = [&](uint64_t *bar) {     // this warp's shared-memory writes and TMEM reads are done: one arrival per warp
            fence_async_smem();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(bar);
        };

        uint32_t ph_in = 0u, ph_out = 0u;
        a_fetch();
        a_store();
        publish(&bars[3]);
        a_fetch();
        for (int h = h0; h <= y_end; ++h) {
            mbar_wait(&bars[1], ph_in);                         // in(h) complete: T1 holds row h, the LN stage is free
            ph_in ^= 1u;
            tc_fence_after();
            if (h - 2 >= y_begin) res_fetch();                  // row h-2: E3(h-2) runs after this iteration's barrier
            e1(h, h + 1 <= y_end);
            publish(&bars[3]);
            if (h + 2 <= y_end) a_fetch();                      // row h+2
            asm volatile("bar.sync 1, %0;" ::"n"(FF_EPI_WARPS * 32) : "memory");      // ring row h complete, readers of row h-3 done
            const int y = h - 1;
            if (y >= y_begin) {
                if (y - 1 >= y_begin) {
                    mbar_wait(&bars[2], ph_out);                // out(y-1) complete: T3 holds row y-1, the dw stage is free
                    ph_out ^= 1u;
                    tc_fence_after();
                    e3();
                }
                dw(y);
                publish(&bars[4]);
            }
        }
        res_fetch();
        mbar_wait(&bars[2], ph_out);
        tc_fence_after();
        e3();
    }
    tc_fence_before();
    __syncthreads();
    if (warp == FF_EPI_WARPS) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_d), "n"(256) : "memory");
    }
}

}  // namespace tc

// ------------------------------------------------------------------------------------ conv_in
// F.pad(reflect, bottom/right to a multiple of 8 -- or the wrapper's centred pad) + Conv2d(3, 31, 3,
// padding=1, bias=False) (MST_Plus_Plus.py:284-289) -> fp32 [B, Hp, Wp, 32].
struct ConvInP {
    const void *in; int in_u8;     // [B, H, W, 3] float32 in [0,1] or uint8 (/255: predict_torch.py:12-19)
    float *out;                    // [B, Hp, Wp, 32]
    const float *w;                // [27][32]: (ky*3+kx)*3+ci major, co minor
    int B, H, W, Hp, Wp, top, left;
};
__device__ __forceinline__ int reflect_idx(int i, int n) {   // torch 'reflect' == REFLECT_101
    if (i < 0) i = -i;
    if (i >= n) i = 2 * n - 2 - i;
    return i;
}
// One thread per output pixel: its 27 inputs (reflect padding of the frame, zero padding of the
// conv) are gathered once into registers, then all 32 output channels are accumulated from
// broadcast float4 weight reads; eight 16-byte stores write the pixel's channel vector.
__global__ void __launch_bounds__(128) conv_in_kernel(const __grid_constant__ ConvInP p) {
    pdl_wait();
    __shared__ __align__(16) float ws[27 * 32];
    for (int i = threadIdx.x; i < 27 * 32; i += blockDim.x) ws[i] = __ldg(p.w + i);
    __syncthreads();
    const long long npx = (long long)p.B * p.Hp * p.Wp;
    const long long px = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (px >= npx) return;
    const int x = (int)(px % p.Wp);
    const long long t = px / p.Wp;
    const int y = (int)(t % p.Hp), b = (int)(t / p.Hp);
    float in[27];
#pragma unroll
    for (int ky = 0; ky < 3; ++ky)
#pragma unroll
        for (int kx = 0; kx < 3; ++kx) {
            const int yp = y + ky - 1, xp = x + kx - 1;          // coordinates in the PADDED image
            const bool inside = (unsigned)yp < (unsigned)p.Hp && (unsigned)xp < (unsigned)p.Wp;   // conv zero padding
            const int ys = reflect_idx(yp - p.top, p.H), xs = reflect_idx(xp - p.left, p.W);
            const long long o = (((long long)b * p.H + min(max(ys, 0), p.H - 1)) * p.W + min(max(xs, 0), p.W - 1)) * 3;
#pragma unroll
            for (int ci = 0; ci < 3; ++ci) {
                float v = 0.f;
                if (inside) v = p.in_u8 ? __fdiv_rn((float)((const uint8_t *)p.in)[o + ci], 255.0f) : ((const float *)p.in)[o + ci];
                in[(ky * 3 + kx) * 3 + ci] = v;
            }
        }
    float *dst = p.out + px * 32;
#pragma unroll
    for (int c4 = 0; c4 < 8; ++c4) {
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int k = 0; k < 27; ++k) {
            const float4 w = *reinterpret_cast<const float4 *>(&ws[k * 32 + 4 * c4]);
            acc.x = fmaf(in[k], w.x, acc.x); acc.y = fmaf(in[k], w.y, acc.y);
            acc.z = fmaf(in[k], w.z, acc.z); acc.w = fmaf(in[k], w.w, acc.w);
        }
        reinterpret_cast<float4 *>(dst)[c4] = acc;      // channel 31 has zero weights -> padded channel stays 0
    }
}

// ------------------------------------------------------------------------------------ depthwise 3x3
// Conv2d(C, C, 3, 1, 1, groups=C, bias=False) on channels-last bf16, optional GELU on the result
// (pos_emb: dw -> GELU -> dw, MST_Plus_Plus.py:104-108; FFN: GELU -> dw -> GELU, :146-153).
struct DwP {
    const bf16 *in; int ldi;
    bf16 *out; int ldo;
    const float *w;               // [9][Cp]
    int B, H, W, Cp, gelu_out, seg;
};
// Thread = (image, column x, group of CPT channels); it walks down a segment of rows keeping the
// 3 x 3 x CPT input window (fp32) and its 9 x CPT weights in registers: three vector loads per
// output instead of nine plus the weight loads.  CPT = 4 keeps the register count low enough for
// 5 CTAs per SM (the 8-channel variant ran at 2 and was latency bound).
#ifndef DW_CPT
#define DW_CPT 4
#endif
template <int CPT> struct DwVec;
template <> struct DwVec<8> { typedef uint4 T; };
template <> struct DwVec<4> { typedef uint2 T; };
template <int CPT>
__device__ __forceinline__ void dw_unpack(const typename DwVec<CPT>::T &raw, float (&f)[CPT]) {
    const __nv_bfloat162 *h2 = reinterpret_cast<const __nv_bfloat162 *>(&raw);
#pragma unroll
    for (int q = 0; q < CPT / 2; ++q) { f[2 * q] = __low2float(h2[q]); f[2 * q + 1] = __high2float(h2[q]); }
}
// Round 2: packed f16 arithmetic.  The bf16 rows are converted to f16 pairs as they are loaded (exact: f16 has more mantissa
// bits, and hidden activations are far inside its range; the conversion saturates), the nine taps accumulate with HFMA2 (11
// mantissa bits through the sum -- less rounding than the bf16 store that follows), GELU as tc::gelu_h2 (defined with the fused
// feed-forward kernel above): 15 instead of 41 instructions per element.
__device__ __forceinline__ uint32_t dw_bf2_to_h2(uint32_t v) {    // two bf16 -> two f16
    uint32_t r;
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(__uint_as_float(v & 0xffff0000u)), "f"(__uint_as_float(v << 16)));
    return r;
}
#ifndef DW_MINB
#define DW_MINB 7        // measured over a forward (nine launches): 7 -> 0.231 ms, 10 -> 0.270, 12 -> 0.346
#endif
template <int CPT>
__global__ void __launch_bounds__(128, DW_MINB) dwconv_kernel(const __grid_constant__ DwP p) {
    static_assert(CPT == 4, "one uint2 (four bf16 channels) per load");
    pdl_wait();
    const int groups = p.Cp / CPT;
    const int segs = (p.H + p.seg - 1) / p.seg;
    const long long total = (long long)p.B * segs * p.W * groups;
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    const int g = (int)(idx % groups);
    long long t = idx / groups;
    const int x = (int)(t % p.W);
    t /= p.W;
    const int sg = (int)(t % segs), b = (int)(t / segs);
    const int y0 = sg * p.seg, y1 = min(p.H, y0 + p.seg);

    __half2 w[9][2];
#pragma unroll
    for (int k = 0; k < 9; ++k) {
        const float4 w0 = __ldg(reinterpret_cast<const float4 *>(p.w + k * p.Cp + CPT * g));
        w[k][0] = __floats2half2_rn(w0.x, w0.y);
        w[k][1] = __floats2half2_rn(w0.z, w0.w);
    }
    // running pointers: rin -> (row being loaded, column x), advanced by one row pitch per load_row
    const long long in_pitch = (long long)p.W * p.ldi, out_pitch = (long long)p.W * p.ldo;
    const bf16 *rin = p.in + (((long long)b * p.H + (y0 - 1)) * p.W + x) * p.ldi + CPT * g;
    bf16 *rout = p.out + (((long long)b * p.H + y0) * p.W + x) * p.ldo + CPT * g;
    const int ldi = p.ldi;
    const bool has_l = x > 0, has_r = x + 1 < p.W;
    int y_next = y0 - 1;                                              // row rin points at
    auto load_row = [&](uint2 (&raw)[3]) {
        raw[0] = raw[1] = raw[2] = make_uint2(0u, 0u);                // conv zero padding
        if ((unsigned)y_next < (unsigned)p.H) {
            if (has_l) raw[0] = __ldg(reinterpret_cast<const uint2 *>(rin - ldi));
            raw[1] = __ldg(reinterpret_cast<const uint2 *>(rin));
            if (has_r) raw[2] = __ldg(reinterpret_cast<const uint2 *>(rin + ldi));
        }
        rin += in_pitch;
        ++y_next;
    };
    auto unpack = [&](const uint2 (&raw)[3], uint32_t (&dst)[3][2]) {
#pragma unroll
        for (int d = 0; d < 3; ++d) { dst[d][0] = dw_bf2_to_h2(raw[d].x); dst[d][1] = dw_bf2_to_h2(raw[d].y); }
    };
    uint32_t win[3][3][2];            // [row slot][dx][channel pair] as f16x2
    uint2 raw[3];
    load_row(raw);
    unpack(raw, win[0]);
    load_row(raw);
    unpack(raw, win[1]);
    load_row(raw);
    for (int yb = y0; yb < y1; yb += 3) {
#pragma unroll
        for (int ph = 0; ph < 3; ++ph) {           // static rotation of the three row slots
            const int y = yb + ph;
            if (y < y1) {
                unpack(raw, win[(ph + 2) % 3]);    // row y + 1
                if (y + 1 < y1) load_row(raw);
                __half2 a0, a1;
#pragma unroll
                for (int ky = 0; ky < 3; ++ky)
#pragma unroll
                    for (int kx = 0; kx < 3; ++kx) {
                        const __half2 v0 = *reinterpret_cast<const __half2 *>(&win[(ph + ky) % 3][kx][0]);
                        const __half2 v1 = *reinterpret_cast<const __half2 *>(&win[(ph + ky) % 3][kx][1]);
                        if (ky == 0 && kx == 0) { a0 = __hmul2(v0, w[0][0]); a1 = __hmul2(v1, w[0][1]); }
                        else { a0 = __hfma2(v0, w[ky * 3 + kx][0], a0); a1 = __hfma2(v1, w[ky * 3 + kx][1], a1); }
                    }
                if (p.gelu_out) { a0 = tc::gelu_h2(a0); a1 = tc::gelu_h2(a1); }
                const float2 f0 = __half22float2(a0), f1 = __half22float2(a1);
                *reinterpret_cast<uint2 *>(rout) = make_uint2(pack_bf16(f0.x, f0.y), pack_bf16(f1.x, f1.y));
                rout += out_pitch;
            }
        }
    }
}

// ------------------------------------------------------------------------------------ fused positional embedding
// pos_emb(v) = dw3x3(GELU(dw3x3(v)))  (MST_Plus_Plus.py:104-108) in ONE kernel: a CTA owns a 16 x 8 pixel tile
// of 32 channels, stages v with a 2-pixel halo in shared memory, evaluates the first conv + GELU on the
// tile plus a 1-pixel halo (rounded to bf16 exactly where the two-kernel pipeline stored it; zero outside
// the map -- that is the second conv's padding) and the second conv from there.  The intermediate map
// never goes to HBM and one launch per attention block disappears.
struct DwPosP {
    const bf16 *in; int ldi;
    bf16 *out; int ldo;
    const float *w1, *w2;         // [9][Cp]
    int B, H, W, Cp;
};
constexpr int DP_TX = 16, DP_TY = 8, DP_CB = 32;
constexpr int DP_IW = DP_TX + 4, DP_IH = DP_TY + 4, DP_MW = DP_TX + 2, DP_MH = DP_TY + 2;
constexpr int DP_SMEM = (DP_IH * DP_IW + DP_MH * DP_MW) * DP_CB * 2 + 2 * 9 * DP_CB * 2;
// One tile by a CTA of NT threads (NT a multiple of 8); smem: DP_SMEM bytes, 16-byte aligned.  Round 2: the tile is
// converted to f16 when it is staged and both convolutions run as packed HFMA2 (a nine-term f16 sum carries 11 mantissa
// bits, more than the bf16 the intermediate map used to be rounded to), GELU as gelu_h2: a third of the instructions of
// the fp32 form (which unpacked every bf16 operand on the ALU pipe).
__device__ __forceinline__ uint32_t h2_to_bf2(__half2 h) {
    const float2 f = __half22float2(h);
    return pack_bf16(f.x, f.y);
}
template <int NT>
__device__ __forceinline__ void dwpos_tile(const DwPosP &p, int bx, int by, int bz, uint8_t *smem) {
    constexpr int IW = DP_IW, IH = DP_IH, MW = DP_MW, MH = DP_MH;
    __half (*sin)[DP_CB] = reinterpret_cast<__half (*)[DP_CB]>(smem);
    __half (*smid)[DP_CB] = reinterpret_cast<__half (*)[DP_CB]>(smem + IH * IW * DP_CB * 2);
    __half (*sw)[9][DP_CB] = reinterpret_cast<__half (*)[9][DP_CB]>(smem + (IH * IW + MH * MW) * DP_CB * 2);
    const int tid = threadIdx.x;
    const int cblocks = p.Cp / DP_CB;
    const int b = bz / cblocks, c0 = (bz - b * cblocks) * DP_CB;
    const int x0 = bx * DP_TX, y0 = by * DP_TY;
    for (int i = tid; i < 2 * 9 * DP_CB; i += NT) {
        const int which = i / (9 * DP_CB), r = i - which * 9 * DP_CB, t = r / DP_CB, c = r - t * DP_CB;
        sw[which][t][c] = __float2half_rn(__ldg((which ? p.w2 : p.w1) + t * p.Cp + c0 + c));
    }
    // stage v: (IH x IW) pixels x 32 channels = 4 x 16-byte vectors per pixel, zeros outside the map
    for (int i = tid; i < IH * IW * 4; i += NT) {
        const int px = i >> 2, q = i & 3;
        const int yy = y0 - 2 + px / IW, xx = x0 - 2 + px % IW;
        uint4 v = make_uint4(0u, 0u, 0u, 0u);
        if ((unsigned)yy < (unsigned)p.H && (unsigned)xx < (unsigned)p.W) {
            v = __ldg(reinterpret_cast<const uint4 *>(p.in + (((long long)b * p.H + yy) * p.W + xx) * p.ldi + c0) + q);
            v = make_uint4(dw_bf2_to_h2(v.x), dw_bf2_to_h2(v.y), dw_bf2_to_h2(v.z), dw_bf2_to_h2(v.w));
        }
        reinterpret_cast<uint4 *>(&sin[px][0])[q] = v;
    }
    __syncthreads();
    // a thread keeps its channel group g = tid & 7 through both loops: the nine tap vectors of the running conv live in
    // registers (as half2 pairs) instead of being re-read from shared memory for every pixel
    const int g_fixed = tid & 7;
    __half2 wr[9][2];
    auto load_weights = [&](int which) {
#pragma unroll
        for (int t = 0; t < 9; ++t) {
            const uint2 w = *reinterpret_cast<const uint2 *>(&sw[which][t][4 * g_fixed]);
            wr[t][0] = *reinterpret_cast<const __half2 *>(&w.x);
            wr[t][1] = *reinterpret_cast<const __half2 *>(&w.y);
        }
    };
    auto conv_at = [&](const __half (*src)[DP_CB], int pitch, int px_centre, int g, __half2 &a0, __half2 &a1) {
#pragma unroll
        for (int t = 0; t < 9; ++t) {
            const uint2 raw = *reinterpret_cast<const uint2 *>(&src[px_centre + (t / 3 - 1) * pitch + (t % 3 - 1)][4 * g]);
            const __half2 v0 = *reinterpret_cast<const __half2 *>(&raw.x), v1 = *reinterpret_cast<const __half2 *>(&raw.y);
            if (t == 0) { a0 = __hmul2(v0, wr[0][0]); a1 = __hmul2(v1, wr[0][1]); }
            else { a0 = __hfma2(v0, wr[t][0], a0); a1 = __hfma2(v1, wr[t][1], a1); }
        }
    };
    // first conv + GELU on the tile and its 1-pixel halo
    load_weights(0);
    for (int i = tid; i < MH * MW * 8; i += NT) {
        const int px = i >> 3, g = i & 7;
        const int my = px / MW, mx = px - my * MW;
        const int yy = y0 - 1 + my, xx = x0 - 1 + mx;
        uint2 o = make_uint2(0u, 0u);
        if ((unsigned)yy < (unsigned)p.H && (unsigned)xx < (unsigned)p.W) {
            __half2 a0, a1;
            conv_at(sin, IW, (my + 1) * IW + (mx + 1), g, a0, a1);
            a0 = tc::gelu_h2(a0);
            a1 = tc::gelu_h2(a1);
            o = make_uint2(*reinterpret_cast<const uint32_t *>(&a0), *reinterpret_cast<const uint32_t *>(&a1));
        }
        *reinterpret_cast<uint2 *>(&smid[px][4 * g]) = o;
    }
    __syncthreads();
    // second conv
    load_weights(1);
    for (int i = tid; i < DP_TY * DP_TX * 8; i += NT) {
        const int px = i >> 3, g = i & 7;
        const int ty = px / DP_TX, tx = px - ty * DP_TX;
        const int yy = y0 + ty, xx = x0 + tx;
        if (yy < p.H && xx < p.W) {
            __half2 a0, a1;
            conv_at(smid, MW, (ty + 1) * MW + (tx + 1), g, a0, a1);
            *reinterpret_cast<uint2 *>(p.out + (((long long)b * p.H + yy) * p.W + xx) * p.ldo + c0 + 4 * g) = make_uint2(h2_to_bf2(a0), h2_to_bf2(a1));
        }
    }
}

// ------------------------------------------------------------------------------------ tiled depthwise 3x3 (coarse-level FFN)
// The row-walking dwconv_kernel above fetches every input pixel three times (left / centre / right neighbour) through
// L1 / L2 and is bound by that latency once its arithmetic is packed f16.  Here a CTA stages a 16 x 8 pixel tile of 32
// channels with its 1-pixel halo in shared memory ONCE (converted to f16 on the way, all of a thread's loads in flight
// together) and evaluates the conv + GELU from there: lane group = 4 channels with their nine taps in registers as half2.
constexpr int DT_IW = DP_TX + 2, DT_IH = DP_TY + 2;
__global__ void __launch_bounds__(256) dwconv_tile_kernel(const __grid_constant__ DwP p) {
    pdl_wait();
    __shared__ __align__(16) __half sin[DT_IH * DT_IW][DP_CB];
    __shared__ __align__(16) __half sw[9][DP_CB];
    const int tid = threadIdx.x;
    const int cblocks = p.Cp / DP_CB;
    const int b = blockIdx.z / cblocks, c0 = (blockIdx.z - b * cblocks) * DP_CB;
    const int x0 = blockIdx.x * DP_TX, y0 = blockIdx.y * DP_TY;
    for (int i = tid; i < 9 * DP_CB; i += 256) sw[i / DP_CB][i % DP_CB] = __float2half_rn(__ldg(p.w + (i / DP_CB) * p.Cp + c0 + i % DP_CB));
    constexpr int NQ = DT_IH * DT_IW * 4, PER = (NQ + 255) / 256;      // 16-byte quads of the staged tile, per thread
    uint4 v[PER];
#pragma unroll
    for (int u = 0; u < PER; ++u) {
        const int i = tid + 256 * u, px = i >> 2, q = i & 3;
        const int yy = y0 - 1 + px / DT_IW, xx = x0 - 1 + px % DT_IW;
        v[u] = make_uint4(0u, 0u, 0u, 0u);                             // zeros outside the map: the conv's padding
        if (i < NQ && (unsigned)yy < (unsigned)p.H && (unsigned)xx < (unsigned)p.W)
            v[u] = __ldg(reinterpret_cast<const uint4 *>(p.in + (((long long)b * p.H + yy) * p.W + xx) * p.ldi + c0) + q);
    }
#pragma unroll
    for (int u = 0; u < PER; ++u) {
        const int i = tid + 256 * u;
        if (i < NQ)
            reinterpret_cast<uint4 *>(&sin[i >> 2][0])[i & 3] = make_uint4(dw_bf2_to_h2(v[u].x), dw_bf2_to_h2(v[u].y), dw_bf2_to_h2(v[u].z), dw_bf2_to_h2(v[u].w));
    }
    __syncthreads();
    const int g = tid & 7;                                             // channel group: fixed per thread (stride 256 keeps it)
    __half2 wr[9][2];
#pragma unroll
    for (int t = 0; t < 9; ++t) {
        const uint2 w = *reinterpret_cast<const uint2 *>(&sw[t][4 * g]);
        wr[t][0] = *reinterpret_cast<const __half2 *>(&w.x);
        wr[t][1] = *reinterpret_cast<const __half2 *>(&w.y);
    }
#pragma unroll
    for (int i = tid; i < DP_TY * DP_TX * 8; i += 256) {
        const int px = i >> 3;
        const int ty = px / DP_TX, tx = px - ty * DP_TX;
        const int yy = y0 + ty, xx = x0 + tx;
        if (yy < p.H && xx < p.W) {
            const int pc = (ty + 1) * DT_IW + (tx + 1);
            __half2 a0, a1;
#pragma unroll
            for (int t = 0; t < 9; ++t) {
                const uint2 raw = *reinterpret_cast<const uint2 *>(&sin[pc + (t / 3 - 1) * DT_IW + (t % 3 - 1)][4 * g]);
                const __half2 v0 = *reinterpret_cast<const __half2 *>(&raw.x), v1 = *reinterpret_cast<const __half2 *>(&raw.y);
                if (t == 0) { a0 = __hmul2(v0, wr[0][0]); a1 = __hmul2(v1, wr[0][1]); }
                else { a0 = __hfma2(v0, wr[t][0], a0); a1 = __hfma2(v1, wr[t][1], a1); }
            }
            if (p.gelu_out) { a0 = tc::gelu_h2(a0); a1 = tc::gelu_h2(a1); }
            *reinterpret_cast<uint2 *>(p.out + (((long long)b * p.H + yy) * p.W + xx) * p.ldo + c0 + 4 * g) = make_uint2(h2_to_bf2(a0), h2_to_bf2(a1));
        }
    }
}

// ------------------------------------------------------------------------------------ attention statistics
// Per image and head: G[i][j] = sum_px k[px][i] q[px][j], nk[i] = sum k^2, nq[j] = sum q^2
// (MST_Plus_Plus.py:127-129: the L2 normalisation runs over ALL pixels, so the reduction is global).
// Accumulation across CTAs is in 64-bit FIXED POINT (2^-24 units, integer atomics): integer addition is
// associative, so the statistics -- and with them the whole forward -- are bit-reproducible from run to
// run; float atomics made two runs differ by 2e-3 of the output range after 15 bf16 layers.
// stats layout per (image, head): 32 x 32 entries; row i < 31, col j < 31: G; [i][31] = nk[i];
// [31][j] = nq[j].
constexpr double STAT_SCALE = 16777216.0;       // 2^24: |sums| < 2^39 fit an int64 with room to spare
struct AttnStatP {
    const bf16 *qkv;     // [B*rows, 3*Cp]: q | k | v
    long long *stats;    // [B][heads][32][32] fixed point (STAT_SCALE), zeroed
    int rows, Cp, heads, px_per_cta;
};
// On the tensor cores (round 2): G = K^T Q over 16 pixels is ONE K-step of mma.sync.m16n8k16 (bf16 operands are exactly
// what q|k|v holds, f32 accumulate), i.e. ~1 warp instruction per pixel, which leaves the statistics bound by reading q and
// k once.  On the CUDA cores a 4x4 register tile of G per thread took 87 warp instructions per pixel (47 us for the 250 K
// pixels of the full-resolution level, 11 % of a forward).
// A head's 31 channels start at column 31*head: the (up to) five aligned 8-channel chunks covering them are staged as a
// 40-wide bf16 window (zero padded to 48), G_window = K_w^T Q_w is 3 x 5 MMA tiles, the head's block is cut out at the
// end; |k_i|^2 and |q_j|^2 are the diagonals of K_w^T K_w / Q_w^T Q_w (the 2 diagonal tiles of every 16-row block).
// Both operands come straight from the [pixel][channel] rows with ldmatrix.trans.  With the fixed-point merge and a split
// of the pixels that depends on the geometry only, the statistics are bit-reproducible and batch invariant.
constexpr int AS_TP = 64, AS_PITCH = 56;          // pixels per staging round; bf16 per staged row (112 B = 7 x 16 B: conflict-free ldmatrix)
__device__ __forceinline__ void as_ldsm_x4_trans(uint32_t (&r)[4], uint32_t addr) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void as_mma_bf16(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3]) : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
struct AttnStatSmem {
    bf16 qs[2][AS_TP][AS_PITCH];                   // two stages: cp.async of round r+1 while round r multiplies
    bf16 ks[2][AS_TP][AS_PITCH];
    float Gs[48][40];                              // window Gram, summed over the CTA's warps in a fixed order
    float Ds[2][48];                               // diagonals: |k|^2, |q|^2
};
// one CTA of 128 threads: pixels [bx * px_per_cta, ...) of (image b, head)
__device__ __forceinline__ void attn_stats_cta(const AttnStatP &p, int bx, int head, int b, AttnStatSmem &S) {
    bf16 (*qs)[AS_TP][AS_PITCH] = S.qs;
    bf16 (*ks)[AS_TP][AS_PITCH] = S.ks;
    float (*Gs)[40] = S.Gs;
    float (*Ds)[48] = S.Ds;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int g = lane >> 2, t = lane & 3;
    const int p0 = bx * p.px_per_cta, p1 = min(p.rows, p0 + p.px_per_cta);
    const int ld = 3 * p.Cp;
    const int lo8 = (head * NF) & ~7, off = head * NF - lo8;
    for (int e = tid; e < 2 * AS_TP * AS_PITCH / 2; e += 128) {      // pad columns (and chunks beyond Cp) stay zero for the whole kernel
        reinterpret_cast<uint32_t *>(&qs[0][0][0])[e] = 0u;
        reinterpret_cast<uint32_t *>(&ks[0][0][0])[e] = 0u;
    }
    for (int e = tid; e < 48 * 40; e += 128) (&Gs[0][0])[e] = 0.f;
    if (tid < 96) (&Ds[0][0])[tid] = 0.f;
    float accG[3][5][4], accK[3][2][4], accQ[3][2][4];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
#pragma unroll
        for (int j = 0; j < 5; ++j)
#pragma unroll
            for (int c = 0; c < 4; ++c) accG[i][j][c] = 0.f;
#pragma unroll
        for (int j = 0; j < 2; ++j)
#pragma unroll
            for (int c = 0; c < 4; ++c) accK[i][j][c] = accQ[i][j][c] = 0.f;
    }
    __syncthreads();
    const uint32_t qs_sh = tc::smem_u32(&qs[0][0][0]), ks_sh = tc::smem_u32(&ks[0][0][0]);
    constexpr uint32_t STAGE = AS_TP * AS_PITCH * 2;                 // bytes per stage of one operand
    // ldmatrix.trans lane roles.  A fragment (16 channels x 16 pixels) of tile mt: matrices (px 0-7 | 8-15) x (ch +0 | +8):
    //   matrix mi = lane >> 3: pixel row (lane & 7) + 8 (mi >> 1), channel 16 mt + 8 (mi & 1)  -> a0..a3
    // B fragments (16 pixels x 8 channels) of tiles nt, nt+1: pixel row (lane & 7) + 8 (mi & 1), channel 8 (nt + (mi >> 1))
    const int a_px = (lane & 7) + 8 * (lane >> 4), a_ch = 8 * ((lane >> 3) & 1);
    const int b_px = (lane & 7) + 8 * ((lane >> 3) & 1), b_ch = 8 * (lane >> 4);
    auto stage_round = [&](int t0, int st) {                          // 16-byte cp.async per (pixel, chunk); rows past the end are zero filled
        for (int e = tid; e < AS_TP * 10; e += 128) {
            const int px = e / 10, c = e - px * 10;
            const int isk = c >= 5, chunk = c - 5 * isk, col0 = lo8 + 8 * chunk;
            if (col0 >= p.Cp) continue;
            const bool live = t0 + px < p1;
            const bf16 *src = p.qkv + ((long long)b * p.rows + (live ? t0 + px : p0)) * ld + isk * p.Cp + col0;
            const uint32_t dst = (isk ? ks_sh : qs_sh) + st * STAGE + 2u * (uint32_t)(px * AS_PITCH + 8 * chunk);
            const int bytes = live ? 16 : 0;
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(bytes) : "memory");
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    const int n_rounds = (p1 - p0 + AS_TP - 1) / AS_TP;
    if (n_rounds > 0) stage_round(p0, 0);
    for (int r = 0; r < n_rounds; ++r) {
        if (r + 1 < n_rounds) {
            stage_round(p0 + (r + 1) * AS_TP, (r + 1) & 1);
            asm volatile("cp.async.wait_group 1;" ::: "memory");
        } else {
            asm volatile("cp.async.wait_group 0;" ::: "memory");
        }
        __syncthreads();
        {
            const uint32_t qb = qs_sh + (r & 1) * STAGE, kb = ks_sh + (r & 1) * STAGE;
            const int r0 = 16 * warp;                               // this warp's 16 pixels of the round
            uint32_t aK[3][4], aQ[3][4], bQ[6][2], bK[6][2];
#pragma unroll
            for (int mt = 0; mt < 3; ++mt) {
                as_ldsm_x4_trans(aK[mt], kb + 2u * (uint32_t)((r0 + a_px) * AS_PITCH + 16 * mt + a_ch));
                as_ldsm_x4_trans(aQ[mt], qb + 2u * (uint32_t)((r0 + a_px) * AS_PITCH + 16 * mt + a_ch));
            }
#pragma unroll
            for (int n2 = 0; n2 < 3; ++n2) {
                uint32_t r4[4];
                as_ldsm_x4_trans(r4, qb + 2u * (uint32_t)((r0 + b_px) * AS_PITCH + 16 * n2 + b_ch));
                bQ[2 * n2][0] = r4[0]; bQ[2 * n2][1] = r4[1]; bQ[2 * n2 + 1][0] = r4[2]; bQ[2 * n2 + 1][1] = r4[3];
                as_ldsm_x4_trans(r4, kb + 2u * (uint32_t)((r0 + b_px) * AS_PITCH + 16 * n2 + b_ch));
                bK[2 * n2][0] = r4[0]; bK[2 * n2][1] = r4[1]; bK[2 * n2 + 1][0] = r4[2]; bK[2 * n2 + 1][1] = r4[3];
            }
#pragma unroll
            for (int mt = 0; mt < 3; ++mt) {
#pragma unroll
                for (int nt = 0; nt < 5; ++nt) as_mma_bf16(accG[mt][nt], aK[mt], bQ[nt][0], bQ[nt][1]);
#pragma unroll
                for (int d = 0; d < 2; ++d) {                       // the two 8-column tiles on the diagonal of row block mt
                    as_mma_bf16(accK[mt][d], aK[mt], bK[2 * mt + d][0], bK[2 * mt + d][1]);
                    as_mma_bf16(accQ[mt][d], aQ[mt], bQ[2 * mt + d][0], bQ[2 * mt + d][1]);
                }
            }
        }
        __syncthreads();                                             // the stage is overwritten by the copies issued next round
    }
    // fragment (row g / g+8, columns 2t, 2t+1) of tile (mt, nt) -> window matrix; warps add in the fixed order 0,1,2,3
    for (int w = 0; w < 4; ++w) {
        if (warp == w) {
#pragma unroll
            for (int mt = 0; mt < 3; ++mt) {
#pragma unroll
                for (int nt = 0; nt < 5; ++nt)
#pragma unroll
                    for (int c = 0; c < 4; ++c) Gs[16 * mt + g + 8 * (c >> 1)][8 * nt + 2 * t + (c & 1)] += accG[mt][nt][c];
#pragma unroll
                for (int d = 0; d < 2; ++d)
#pragma unroll
                    for (int c = 0; c < 4; ++c) {
                        const int row = g + 8 * (c >> 1), col = 8 * d + 2 * t + (c & 1);     // inside the 16 x 16 diagonal block
                        if (row == col) { Ds[0][16 * mt + row] += accK[mt][d][c]; Ds[1][16 * mt + row] += accQ[mt][d][c]; }
                    }
            }
        }
        __syncthreads();
    }
    unsigned long long *out = reinterpret_cast<unsigned long long *>(p.stats) + ((long long)b * p.heads + head) * 1024;
    for (int e = tid; e < 1024; e += 128) {
        const int i = e >> 5, j = e & 31;
        float v;
        if (i < NF && j < NF) v = Gs[off + i][off + j];
        else if (i < NF) v = Ds[0][off + i];                                                  // [i][31] = |k_i|^2
        else if (j < NF) v = Ds[1][off + j];                                                  // [31][j] = |q_j|^2
        else v = 0.f;
        atomicAdd(out + e, (unsigned long long)__double2ll_rn((double)v * STAT_SCALE));
    }
}

// attn = softmax_j(rescale * G_ij / (max(|k_i|,1e-12) max(|q_j|,1e-12)))  (:127-131), then
// M[co][h*31+j] = sum_i Wproj[co][h*31+i] attn_h[i][j]  -> bf16 [B][Cp][Cp] (zero padded).
struct AttnFinP {
    const long long *stats; const float *rescale; const float *wproj;   // wproj fp32 [c][c]
    bf16 *M;             // [B][Cp][Cp]
    int c, Cp, heads;
};
// ------------------------------------------------------------------------------------ attention side kernel
// Everything between the q|k|v GEMM and the projection GEMM of an MSAB in ONE launch of heterogeneous CTAs (128 threads):
//   blocks [0, nA)   statistics (attn_stats_cta); the LAST statistics CTA of an (image, head) -- a ticket counter behind
//                    a __threadfence -- turns the finished sums into that head's softmax and its 31 columns of
//                    M = Wproj . blockdiag(attn)
//   blocks [nA, ..)  positional-embedding tiles (dwpos_tile), which depend on v only
// The two parts are independent (one reads q|k and is bound by HBM, the other is CUDA-core work on v), so they overlap
// on the SMs instead of running back to back, and two launches per block disappear.  Which CTA finalises is a race, what
// it computes is not: the sums are integers (fixed point) and the finalising arithmetic has one fixed order.
struct AttnSideP {
    AttnStatP st;
    AttnFinP fin;
    DwPosP dp;
    unsigned *tickets;      // [B][heads], zeroed by the q|k|v GEMM together with the statistics
    int ctasA, nA, gx, gy;  // statistics CTAs per (image, head), their total; positional-embedding grid (x, y)
};
union AttnSideSmem {
    AttnStatSmem st;
    uint8_t dp[DP_SMEM];
};
// wsm: the head's 31 columns of Wproj, [c][32] floats (staged here with coalesced loads while the softmax rows are computed)
__device__ __forceinline__ void attn_finalize_head(const AttnFinP &p, int b, int h, float (*attn)[32], float *rq, float (*wsm)[32]) {
    const int tid = threadIdx.x;
    const long long *S = p.stats + ((long long)b * p.heads + h) * 1024;
    for (int e0 = tid; e0 < p.c * 32; e0 += 128 * 8) {          // eight loads in flight per thread: this CTA runs alone, latency is all there is
        float v[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const int e = e0 + 128 * u, co = e >> 5, i = e & 31;
            v[u] = (e < p.c * 32 && i < NF) ? __ldg(p.wproj + (long long)co * p.c + h * NF + i) : 0.f;
        }
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const int e = e0 + 128 * u;
            if (e < p.c * 32) wsm[e >> 5][e & 31] = v[u];
        }
    }
    // fixed point -> float: int64 -> float rounds once and the scale is a power of two, the same bits as the detour through double
    constexpr float INV_SCALE = (float)(1.0 / STAT_SCALE);
    if (tid < 32) rq[tid] = tid < NF ? 1.0f / fmaxf(sqrtf((float)__ldcg(S + 31 * 32 + tid) * INV_SCALE), 1e-12f) : 0.f;
    __syncthreads();
    if (tid < NF) {          // softmax row i = tid
        const int i = tid;
        const float sc = __ldg(p.rescale + h) / fmaxf(sqrtf((float)__ldcg(S + i * 32 + 31) * INV_SCALE), 1e-12f);
        float row[NF], mx = -INFINITY;
#pragma unroll
        for (int j = 0; j < NF; ++j) {
            row[j] = ((float)__ldcg(S + i * 32 + j) * INV_SCALE) * (sc * rq[j]);
            mx = fmaxf(mx, row[j]);
        }
        float sum = 0.f;
#pragma unroll
        for (int j = 0; j < NF; ++j) { row[j] = __expf(row[j] - mx); sum += row[j]; }
        const float inv = 1.0f / sum;
#pragma unroll
        for (int j = 0; j < NF; ++j) attn[i][j] = row[j] * inv;
    }
    __syncthreads();
    bf16 *M = p.M + (long long)b * p.Cp * p.Cp;
    // element e = (row co = e / 32, column j = e % 32) of the head's block; a thread's elements e, e + 128, e + 256, e + 384 share
    // their column and sit four rows apart: four independent accumulation chains (each in the fixed order i = 0 .. 30)
    for (int e0 = tid; e0 < p.Cp * 32; e0 += 512) {
        const int co0 = e0 >> 5, j = e0 & 31;
        if (j < NF) {
            float v[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
            for (int i = 0; i < NF; ++i) {
                const float a = attn[i][j];
#pragma unroll
                for (int u = 0; u < 4; ++u) v[u] = fmaf(wsm[min(co0 + 4 * u, p.c - 1)][i], a, v[u]);
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int co = co0 + 4 * u;
                M[(long long)co * p.Cp + h * NF + j] = __float2bfloat16_rn(co < p.c ? v[u] : 0.f);
            }
        } else if (h == p.heads - 1) {
#pragma unroll
            for (int u = 0; u < 4; ++u)
                for (int k = p.c; k < p.Cp; ++k) M[(long long)(co0 + 4 * u) * p.Cp + k] = __float2bfloat16_rn(0.f);     // padded columns
        }
    }
}
#ifndef AVB_SIDE_MINB
#define AVB_SIDE_MINB 4      // resident CTAs per SM the register allocation aims at
#endif
__global__ void __launch_bounds__(128, AVB_SIDE_MINB) attn_side_kernel(const __grid_constant__ AttnSideP p) {
    pdl_wait();
    __shared__ __align__(16) AttnSideSmem sm;
    __shared__ int is_last;
    const int bid = blockIdx.x;
    if (bid >= p.nA) {
        const int r = bid - p.nA;
        const int bx = r % p.gx, q = r / p.gx;
        dwpos_tile<128>(p.dp, bx, q % p.gy, q / p.gy, sm.dp);
        return;
    }
    const int bx = bid % p.ctasA, q = bid / p.ctasA;
    const int head = q % p.st.heads, b = q / p.st.heads;
    attn_stats_cta(p.st, bx, head, b, sm.st);
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) is_last = atomicAdd(p.tickets + b * p.st.heads + head, 1u) == (unsigned)(p.ctasA - 1);
    __syncthreads();
    if (!is_last) return;
    __threadfence();
    static_assert(sizeof(sm.st.qs) + sizeof(sm.st.ks) >= 124 * 32 * sizeof(float), "Wproj column block fits the staging buffers");
    attn_finalize_head(p.fin, b, head, reinterpret_cast<float (*)[32]>(&sm.st.Gs[0][0]), &sm.st.Ds[0][0],
                       reinterpret_cast<float (*)[32]>(&sm.st.qs[0][0][0]));
}

// ------------------------------------------------------------------------------------ band projection
// out[px][r] = sum_b cube[px][b] * w[r][b]  (uv_helpers.py:142-146 integrate_band / np.tensordot;
// mantis_shrimp.py:49-60 uses ten such bands).  fp32, one thread per (pixel, receptor).
__global__ void __launch_bounds__(256) band_project_kernel(const float *__restrict__ cube, const float *__restrict__ w, float *__restrict__ out,
                                                           long long npx, int nb, int nr) {
    extern __shared__ float wsm[];
    for (int i = threadIdx.x; i < nb * nr; i += blockDim.x) wsm[i] = __ldg(w + i);
    __syncthreads();
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < npx * nr; e += (long long)gridDim.x * blockDim.x) {
        const long long px = e / nr;
        const int r = (int)(e - px * nr);
        const float *c = cube + px * nb;
        float acc = 0.f;
        for (int k = 0; k < nb; ++k) acc = fmaf(__ldg(c + k), wsm[r * nb + k], acc);
        out[e] = acc;
    }
}

// ------------------------------------------------------------------------------------ safe_norm
// uv_helpers.py:47-53 safe_norm: (x - min) / (max - min) over a whole map, zeros when the range is
// below 1e-9.  Maps are interleaved: element px of map k is in[px * stride + k].
__device__ __forceinline__ uint32_t f2ord(float f) {          // order-preserving float -> uint
    const uint32_t u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float ord2f(uint32_t o) {
    return __uint_as_float((o & 0x80000000u) ? (o & 0x7fffffffu) : ~o);
}
__global__ void __launch_bounds__(256) minmax_kernel(const float *__restrict__ in, long long npx, int stride, int n_maps, uint32_t *mm) {
    const int k = blockIdx.y;
    float mn = INFINITY, mx = -INFINITY;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < npx; i += (long long)gridDim.x * blockDim.x) {
        const float v = __ldg(in + i * stride + k);
        mn = fminf(mn, v); mx = fmaxf(mx, v);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
        mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    }
    if ((threadIdx.x & 31) == 0) {
        atomicMin(mm + k, f2ord(mn));
        atomicMax(mm + n_maps + k, f2ord(mx));
    }
}
__global__ void __launch_bounds__(256) safe_norm_kernel(const float *__restrict__ in, float *__restrict__ out, long long npx, int stride,
                                                        int n_maps, const uint32_t *mm) {
    const int k = blockIdx.y;
    const float mn = ord2f(mm[k]), mx = ord2f(mm[n_maps + k]);
    const double range = (double)mx - (double)mn;              // python floats in the reference
    const float den = (float)range;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < npx; i += (long long)gridDim.x * blockDim.x) {
        const float v = __ldg(in + i * stride + k);
        out[i * stride + k] = range < 1e-9 ? 0.f : __fdiv_rn(__fsub_rn(v, mn), den);
    }
}

// ------------------------------------------------------------------------------------ host: weights
struct MsabW {
    int c, Cp, heads, Hp;
    const float *rescale, *wproj_f32, *bproj, *ln_g, *ln_b;       // device fp32
    const float *pos0, *pos2, *ffn_dw;                            // device fp32 [9][Cp] / [9][Hp]
    const bf16 *wqkv, *ffn0, *ffn4;                               // device bf16
    const float *wqkv32;                                          // device fp32 [3*Cp][Cp] (tf32 TMA kernel)
    const uint8_t *ffn_blob;                                      // fused FFN (Cp == 32): per 128-channel hidden chunk W0 | W4
};
struct BodyW {
    const bf16 *embedding, *mapping;     // [32][9*32]
    MsabW enc[2], bott, dec[2];
    const bf16 *down[2];                 // [Cp_out][16*Cp_in]
    const bf16 *up[2];                   // [4*Cp_out][Cp_in]
    const float *up_bias[2];             // [4*Cp_out]
    const bf16 *fuse[2];                 // [Cp_out][2*Cp_out]
};
struct Model {
    int device;
    void *blob;                          // one device allocation holding every tensor below
    const float *conv_in;                // [27][32]
    BodyW body[3];
    const bf16 *conv_out;                // [32][9*32]
};

// Builder: appends host-side tensors to one staging buffer (256-byte aligned each) and records
// where the device pointer must be patched once the blob is uploaded.
struct Packer {
    std::vector<uint8_t> host;
    struct Fix { const void **slot; size_t off; };
    std::vector<Fix> fixes;
    size_t reserve(size_t bytes) {
        const size_t off = (host.size() + 255) / 256 * 256;
        host.resize(off + bytes, 0);
        return off;
    }
    float *f32(const void **slot, size_t n) {
        const size_t off = reserve(n * 4);
        fixes.push_back({slot, off});
        return reinterpret_cast<float *>(host.data() + off);
    }
    uint16_t *b16(const void **slot, size_t n) {
        const size_t off = reserve(n * 2);
        fixes.push_back({slot, off});
        return reinterpret_cast<uint16_t *>(host.data() + off);
    }
};
// NOTE: pointers returned by Packer::f32 / b16 are invalidated by the next reserve(); fill each
// tensor right after asking for it, addressing through the offset.

static uint16_t f2bf(float f) {          // round to nearest even
    uint32_t u;
    memcpy(&u, &f, 4);
    if ((u & 0x7fffffffu) > 0x7f800000u) return 0x7fc0;
    u += 0x7fffu + ((u >> 16) & 1u);
    return (uint16_t)(u >> 16);
}

static uint16_t f2h(float f) {           // IEEE half, round to nearest even
    const __half h = __float2half_rn(f);
    uint16_t u;
    memcpy(&u, &h, 2);
    return u;
}

struct Cursor {
    const float *p; int64_t left;
    const float *take(int64_t n) {
        if (n > left) return nullptr;
        const float *r = p; p += n; left -= n;
        return r;
    }
};

#define TAKE(var, n)                                   \
    const float *var = cur.take(n);                    \
    if (!var) return false;

// dense [Cout][Cin] (row-major) -> bf16 [Np][Kp], optional row / column offsets for fused layouts
static void put_dense(uint16_t *dst, int Kp, const float *w, int cout, int cin, int row0, int col0) {
    for (int o = 0; o < cout; ++o)
        for (int i = 0; i < cin; ++i) dst[(size_t)(row0 + o) * Kp + col0 + i] = f2bf(w[(size_t)o * cin + i]);
}

static bool pack_msab(Packer &pk, Cursor &cur, MsabW &m, int c) {
    m.c = c; m.Cp = pad32(c); m.heads = c / NF; m.Hp = pad32(4 * c);
    const int Cp = m.Cp, Hp = m.Hp;
    TAKE(rescale, m.heads);
    TAKE(wq, (int64_t)c * c); TAKE(wk, (int64_t)c * c); TAKE(wv, (int64_t)c * c);
    TAKE(wp, (int64_t)c * c); TAKE(bp, c);
    TAKE(pos0, (int64_t)c * 9); TAKE(pos2, (int64_t)c * 9);
    TAKE(f0, (int64_t)4 * c * c); TAKE(f2, (int64_t)4 * c * 9); TAKE(f4, (int64_t)4 * c * c);
    TAKE(lg, c); TAKE(lb, c);
    { float *d = pk.f32((const void **)&m.rescale, 4); for (int i = 0; i < m.heads; ++i) d[i] = rescale[i]; }
    { float *d = pk.f32((const void **)&m.wproj_f32, (size_t)c * c); memcpy(d, wp, sizeof(float) * c * c); }
    { float *d = pk.f32((const void **)&m.bproj, Cp); for (int i = 0; i < c; ++i) d[i] = bp[i]; }
    { float *d = pk.f32((const void **)&m.ln_g, Cp); for (int i = 0; i < c; ++i) d[i] = lg[i]; }
    { float *d = pk.f32((const void **)&m.ln_b, Cp); for (int i = 0; i < c; ++i) d[i] = lb[i]; }
    // depthwise weights (C,1,3,3) -> [9][Cp]
    { float *d = pk.f32((const void **)&m.pos0, (size_t)9 * Cp); for (int ch = 0; ch < c; ++ch) for (int t = 0; t < 9; ++t) d[t * Cp + ch] = pos0[ch * 9 + t]; }
    { float *d = pk.f32((const void **)&m.pos2, (size_t)9 * Cp); for (int ch = 0; ch < c; ++ch) for (int t = 0; t < 9; ++t) d[t * Cp + ch] = pos2[ch * 9 + t]; }
    { float *d = pk.f32((const void **)&m.ffn_dw, (size_t)9 * Hp); for (int ch = 0; ch < 4 * c; ++ch) for (int t = 0; t < 9; ++t) d[t * Hp + ch] = f2[ch * 9 + t]; }
    // q | k | v stacked along N: rows [0,c), [Cp,Cp+c), [2Cp,2Cp+c)
    { uint16_t *d = pk.b16((const void **)&m.wqkv, (size_t)3 * Cp * Cp);
      put_dense(d, Cp, wq, c, c, 0, 0); put_dense(d, Cp, wk, c, c, Cp, 0); put_dense(d, Cp, wv, c, c, 2 * Cp, 0); }
    { float *d = pk.f32((const void **)&m.wqkv32, (size_t)3 * Cp * Cp);
      const float *src[3] = {wq, wk, wv};
      for (int t = 0; t < 3; ++t)
          for (int r = 0; r < c; ++r)
              for (int k = 0; k < c; ++k) d[(size_t)(t * Cp + r) * Cp + k] = src[t][(size_t)r * c + k]; }
    { uint16_t *d = pk.b16((const void **)&m.ffn0, (size_t)Hp * Cp); put_dense(d, Cp, f0, 4 * c, c, 0, 0); }
    { uint16_t *d = pk.b16((const void **)&m.ffn4, (size_t)Cp * Hp); put_dense(d, Hp, f4, c, 4 * c, 0, 0); }
    m.ffn_blob = nullptr;
    if (Cp == 32) {
        // operands of ffn_fused_kernel, chunk by chunk, in the kernel's shared-memory layout (canonical K-major, 16-byte
        // entries of 8 k values): W0 [Cp/8][128 n][8] bf16, W4 [16][Cp n][8] f16
        const int w0_el = (Cp / 8) * 128 * 8, w4_el = 16 * Cp * 8, chunk_el = w0_el + w4_el;
        const int chunks = Hp / 128;
        uint16_t *d = pk.b16((const void **)&m.ffn_blob, (size_t)chunks * chunk_el);
        for (int ck = 0; ck < chunks; ++ck) {
            uint16_t *w0 = d + (size_t)ck * chunk_el, *w4 = w0 + w0_el;
            for (int kc = 0; kc < Cp / 8; ++kc)
                for (int n = 0; n < 128; ++n)
                    for (int e = 0; e < 8; ++e) {
                        const int hid = ck * 128 + n, ch = kc * 8 + e;
                        w0[(kc * 128 + n) * 8 + e] = (hid < 4 * c && ch < c) ? f2bf(f0[(size_t)hid * c + ch]) : 0;
                    }
            for (int kc = 0; kc < 16; ++kc)
                for (int n = 0; n < Cp; ++n)
                    for (int e = 0; e < 8; ++e) {
                        const int hid = ck * 128 + kc * 8 + e;
                        w4[(kc * Cp + n) * 8 + e] = (hid < 4 * c && n < c) ? f2h(f4[(size_t)n * 4 * c + hid]) : 0;
                    }
        }
    }
    return true;
}

// Conv2d weight (Cout, Cin, kh, kw) -> bf16 [Np][kh*kw*Cp_in], k = (ky*kw+kx)*Cp_in + ci
static void put_conv(uint16_t *dst, const float *w, int cout, int cin, int kh, int kw, int Cpin) {
    const int K = kh * kw * Cpin;
    for (int o = 0; o < cout; ++o)
        for (int i = 0; i < cin; ++i)
            for (int t = 0; t < kh * kw; ++t) dst[(size_t)o * K + t * Cpin + i] = f2bf(w[((size_t)o * cin + i) * kh * kw + t]);
}

static bool pack_model(Packer &pk, Model &M, const float *params, int64_t count) {
    Cursor cur{params, count};
    {
        TAKE(w, 31 * 3 * 9);
        float *d = pk.f32((const void **)&M.conv_in, 27 * 32);
        for (int co = 0; co < 31; ++co)
            for (int ci = 0; ci < 3; ++ci)
                for (int t = 0; t < 9; ++t) d[(t * 3 + ci) * 32 + co] = w[(co * 3 + ci) * 9 + t];
    }
    for (int s = 0; s < 3; ++s) {
        BodyW &B = M.body[s];
        { TAKE(w, 31 * 31 * 9); uint16_t *d = pk.b16((const void **)&B.embedding, (size_t)32 * 288); put_conv(d, w, 31, 31, 3, 3, 32); }
        int c = NF;
        for (int i = 0; i < 2; ++i) {
            if (!pack_msab(pk, cur, B.enc[i], c)) return false;
            TAKE(w, (int64_t)2 * c * c * 16);
            const int Cpi = pad32(c), Cpo = pad32(2 * c);
            uint16_t *d = pk.b16((const void **)&B.down[i], (size_t)Cpo * 16 * Cpi);
            put_conv(d, w, 2 * c, c, 4, 4, Cpi);
            c *= 2;
        }
        if (!pack_msab(pk, cur, B.bott, c)) return false;
        for (int i = 0; i < 2; ++i) {
            const int co = c / 2, Cpi = pad32(c), Cpo = pad32(co);
            TAKE(wt, (int64_t)c * co * 4);       // ConvTranspose2d weight (Cin, Cout, 2, 2)
            TAKE(bt, co);
            TAKE(wf, (int64_t)co * c);           // fusion 1x1 (Cout=co, Cin=c = [up | skip])
            { uint16_t *d = pk.b16((const void **)&B.up[i], (size_t)4 * Cpo * Cpi);
              for (int ci = 0; ci < c; ++ci)
                  for (int o = 0; o < co; ++o)
                      for (int q = 0; q < 4; ++q) d[(size_t)(q * Cpo + o) * Cpi + ci] = f2bf(wt[((size_t)ci * co + o) * 4 + q]); }
            { float *d = pk.f32((const void **)&B.up_bias[i], (size_t)4 * Cpo);
              for (int q = 0; q < 4; ++q) for (int o = 0; o < co; ++o) d[q * Cpo + o] = bt[o]; }
            { uint16_t *d = pk.b16((const void **)&B.fuse[i], (size_t)Cpo * 2 * Cpo);
              for (int o = 0; o < co; ++o) {
                  for (int k = 0; k < co; ++k) d[(size_t)o * 2 * Cpo + k] = f2bf(wf[(size_t)o * c + k]);                 // up half
                  for (int k = 0; k < co; ++k) d[(size_t)o * 2 * Cpo + Cpo + k] = f2bf(wf[(size_t)o * c + co + k]);      // skip half
              } }
            if (!pack_msab(pk, cur, B.dec[i], co)) return false;
            c = co;
        }
        { TAKE(w, 31 * 31 * 9); uint16_t *d = pk.b16((const void **)&B.mapping, (size_t)32 * 288); put_conv(d, w, 31, 31, 3, 3, 32); }
    }
    { TAKE(w, 31 * 31 * 9); uint16_t *d = pk.b16((const void **)&M.conv_out, (size_t)32 * 288); put_conv(d, w, 31, 31, 3, 3, 32); }
    return cur.left == 0;
}

// ------------------------------------------------------------------------------------ host: schedule
struct Workspace {
    float *x0, *hA, *hB, *f0, *f1, *f2, *u1, *u0, *d1, *d0, *xt;
    long long *stats;
    unsigned *tickets;
    bf16 *qkv, *p1, *p2, *ln, *hid1, *hid2, *M;
    size_t bytes;
};
static size_t carve(Workspace *w, uint8_t *base, int B, int Hp, int Wp) {
    const size_t n0 = (size_t)B * Hp * Wp, n1 = n0 / 4, n2 = n0 / 16;
    size_t off = 0;
    auto take = [&](size_t bytes) { const size_t o = off; off += (bytes + 255) / 256 * 256; return base ? base + o : nullptr; };
#define WS_F(name, elems) { float *ptr = (float *)take((elems) * 4); if (w) w->name = ptr; }
#define WS_B(name, elems) { bf16 *ptr = (bf16 *)take((elems) * 2); if (w) w->name = ptr; }
    WS_F(x0, n0 * 32) WS_F(hA, n0 * 32) WS_F(hB, n0 * 32) WS_F(f0, n0 * 32) WS_F(f1, n1 * 64) WS_F(f2, n2 * 128)
    WS_F(u1, n1 * 64) WS_F(u0, n0 * 32) WS_F(d1, n1 * 64) WS_F(d0, n0 * 32) WS_F(xt, n0 * 32)
    { unsigned *ptr = (unsigned *)take((size_t)B * 4 * 4); if (w) w->tickets = ptr; }       // directly in front of stats: cleared together
    { long long *ptr = (long long *)take((size_t)B * 4 * 1024 * 8); if (w) w->stats = ptr; }
    WS_B(qkv, n0 * 96) WS_B(p1, n0 * 32) WS_B(p2, n0 * 32) WS_B(ln, n0 * 32) WS_B(hid1, n0 * 128) WS_B(hid2, n0 * 128)
    WS_B(M, (size_t)B * 128 * 128)
#undef WS_F
#undef WS_B
    if (w) w->bytes = off;
    return off;
}

struct Ctx {
    cudaStream_t st;
    int B;
    int unsupported = 0;      // a layer shape none of the kernels covers (cannot happen for MST++'s own shapes)
};

template <int BN, bool A_BF16, int MODE, bool DEEP>
static void launch_gemm_td(Ctx &cx, const GemmP &p, dim3 grid, const char *name) {
    constexpr int smem = 2 * (BK / 8) * (BM / 8) * 128 + 2 * (BK / 8) * (BN / 8) * 128;
    static SmemOptIn opt_in;              // per instantiation, per device
    opt_in.ensure(tc::gemm_tc_kernel<BN, A_BF16, MODE, DEEP>, smem);
    AVB_TIMED(name, cx.st);
    launch_pdl(tc::gemm_tc_kernel<BN, A_BF16, MODE, DEEP>, grid, dim3(GEMM_THREADS), smem, cx.st, p);
}
template <int BN, bool A_BF16, int MODE>
static void launch_gemm_t(Ctx &cx, const GemmP &p, const char *name) {
    dim3 grid((p.rows + BM - 1) / BM, p.Np / BN, cx.B);
    // fewer than ~3 CTAs per SM: nothing else hides the load latency of the K loop
    if ((long long)grid.x * grid.y * grid.z < 3LL * sm_count()) launch_gemm_td<BN, A_BF16, MODE, true>(cx, p, grid, name);
    else launch_gemm_td<BN, A_BF16, MODE, false>(cx, p, grid, name);
}
template <int BN, int KP, bool A_BF16, bool LN, int EPI>
static void launch_pw_t(Ctx &cx, const GemmP &p, const char *name) {
    constexpr int smem = 2 * (KP / 8) * (BM / 8) * 128 + (KP / 8) * (BN / 8) * 128 + (LN ? 2 * KP * 4 : 0);
    constexpr int tmem_cols = 2 * BN <= 32 ? 32 : (2 * BN <= 64 ? 64 : (2 * BN <= 128 ? 128 : (2 * BN <= 256 ? 256 : 512)));
    static SmemOptIn opt_in;              // per instantiation, per device
    opt_in.ensure(tc::gemm_pw_kernel<BN, KP, A_BF16, LN, EPI>, smem);
    // resident CTAs per SM: TMEM columns, shared memory, and no more than the pipeline needs
    const int per_sm = std::max(1, std::min(std::min(512 / tmem_cols, (200 * 1024) / (smem + 1024)), 4));
    const int m_tiles = (p.rows + BM - 1) / BM, ny = p.Np / BN;
    int gx = std::max(1, std::min(m_tiles, sm_count() * per_sm / std::max(1, ny * cx.B)));
    const int per_cta = (m_tiles + gx - 1) / gx;
    gx = (m_tiles + per_cta - 1) / per_cta;              // same depth, no idle CTAs
    AVB_TIMED(name, cx.st);
    launch_pdl(tc::gemm_pw_kernel<BN, KP, A_BF16, LN, EPI>, dim3(gx, ny, cx.B), dim3(GEMM_THREADS), smem, cx.st, p);
}

// cuTensorMapEncodeTiled through the runtime's driver entry point (no link against libcuda)
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                  const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_tiled_fn() {
    static const EncodeTiledFn fn = [] {             // thread-safe function-local static: resolved exactly once
        void *ptr = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            return reinterpret_cast<EncodeTiledFn>(ptr);
        return static_cast<EncodeTiledFn>(nullptr);
    }();
    return fn;
}

// bf16 activation matrix [total_rows, lda] (K used columns) as {8 channels, rows, K/8}: a box of
// {8, 128, K/8} is one operand tile in canonical K-major layout
static bool make_a_map(CUtensorMap *tm, const bf16 *A, long long total_rows, int lda, int K) {
    EncodeTiledFn enc = encode_tiled_fn();
    if (!enc) return false;
    const cuuint64_t gdim[3] = {8, (cuuint64_t)total_rows, (cuuint64_t)(K / 8)};
    const cuuint64_t gstride[2] = {(cuuint64_t)lda * 2, 16};
    const cuuint32_t box[3] = {8, (cuuint32_t)BM, (cuuint32_t)(K / 8)};
    const cuuint32_t estride[3] = {1, 1, 1};
    return enc(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<bf16 *>(A), gdim, gstride, box, estride, CU_TENSOR_MAP_INTERLEAVE_NONE,
               CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

static bool make_a_map_f32(CUtensorMap *tm, const float *A, long long total_rows, int lda, int K) {
    EncodeTiledFn enc = encode_tiled_fn();
    if (!enc) return false;
    const cuuint64_t gdim[3] = {4, (cuuint64_t)total_rows, (cuuint64_t)(K / 4)};
    const cuuint64_t gstride[2] = {(cuuint64_t)lda * 4, 16};
    const cuuint32_t box[3] = {4, (cuuint32_t)BM, (cuuint32_t)(K / 4)};
    const cuuint32_t estride[3] = {1, 1, 1};
    return enc(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float *>(A), gdim, gstride, box, estride, CU_TENSOR_MAP_INTERLEAVE_NONE,
               CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

template <int BN, int KP, int EPI>
static bool launch_tma32_t(Ctx &cx, const GemmP &p, const char *name) {
    if (!p.W32 || p.K1 < p.K || p.w_bstride != 0 || (reinterpret_cast<uintptr_t>(p.A1) & 15) || (p.lda1 & 3)) return false;
    alignas(64) CUtensorMap tm;
    if (!make_a_map_f32(&tm, static_cast<const float *>(p.A1), (long long)cx.B * p.rows, p.lda1, KP)) return false;
    constexpr int NS = KP <= 32 ? 4 : (KP <= 64 ? 3 : 2);
    constexpr int smem = NS * (KP / 4) * (BM / 8) * 128 + (KP / 4) * (BN / 8) * 128;
    constexpr int tmem_cols = 2 * BN <= 32 ? 32 : (2 * BN <= 64 ? 64 : (2 * BN <= 128 ? 128 : (2 * BN <= 256 ? 256 : 512)));
    static SmemOptIn opt_in;              // per instantiation, per device
    opt_in.ensure(tc::gemm_tma32_kernel<BN, KP, EPI>, smem);
    const int per_sm = std::max(1, std::min(std::min(512 / tmem_cols, (200 * 1024) / (smem + 1024)), 4));
    const int m_tiles = (p.rows + BM - 1) / BM, ny = p.Np / BN;
    int gx = std::max(1, std::min(m_tiles, sm_count() * per_sm / std::max(1, ny * cx.B)));
    const int per_cta = (m_tiles + gx - 1) / gx;
    gx = (m_tiles + per_cta - 1) / per_cta;
    AVB_TIMED(name, cx.st);
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(gx, ny, cx.B); cfg.blockDim = dim3(GEMM_THREADS); cfg.dynamicSmemBytes = smem; cfg.stream = cx.st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, tc::gemm_tma32_kernel<BN, KP, EPI>, p, tm) == cudaSuccess;
}

template <int BN, int KP, int EPI>
static bool launch_tma_t(Ctx &cx, const GemmP &p, const char *name) {
    if (p.K1 < p.K || (reinterpret_cast<uintptr_t>(p.A1) & 15) || (p.lda1 & 7)) return false;
    alignas(64) CUtensorMap tm;
    if (!make_a_map(&tm, static_cast<const bf16 *>(p.A1), (long long)cx.B * p.rows, p.lda1, KP)) return false;
    constexpr int NS = KP <= 64 ? 4 : 3;
    constexpr int smem = NS * (KP / 8) * (BM / 8) * 128 + (KP / 8) * (BN / 8) * 128;
    constexpr int tmem_cols = 2 * BN <= 32 ? 32 : (2 * BN <= 64 ? 64 : (2 * BN <= 128 ? 128 : (2 * BN <= 256 ? 256 : 512)));
    static SmemOptIn opt_in;              // per instantiation, per device
    opt_in.ensure(tc::gemm_tma_kernel<BN, KP, EPI>, smem);
    const int per_sm = std::max(1, std::min(std::min(512 / tmem_cols, (200 * 1024) / (smem + 1024)), 4));
    const int m_tiles = (p.rows + BM - 1) / BM, ny = p.Np / BN;
    int gx = std::max(1, std::min(m_tiles, sm_count() * per_sm / std::max(1, ny * cx.B)));
    const int per_cta = (m_tiles + gx - 1) / gx;
    gx = (m_tiles + per_cta - 1) / per_cta;
    AVB_TIMED(name, cx.st);
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(gx, ny, cx.B); cfg.blockDim = dim3(GEMM_THREADS); cfg.dynamicSmemBytes = smem; cfg.stream = cx.st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, tc::gemm_tma_kernel<BN, KP, EPI>, p, tm) == cudaSuccess;
}

// Shapes of the MST++ pointwise layers that take the pipelined kernel (anything else falls through
// to the generic K-chunked kernel): K = the padded channel count of the level, N a multiple of it.
template <bool A_BF16>
static bool launch_pw(Ctx &cx, const GemmP &p, const char *name) {
    if (p.K1 < p.K && 2 * p.K1 != p.K) return false;
    const bool ln = p.ln_g != nullptr;
    const int epi = tc::epi_of(p);
#define PW_CASE(BN_, KP_, LN_, EPI_) \
    if (p.K == KP_ && p.Np % BN_ == 0 && ln == LN_ && epi == (EPI_)) { launch_pw_t<BN_, KP_, A_BF16, LN_, (EPI_)>(cx, p, name); return true; }
    using namespace tc;
    if constexpr (A_BF16) {
        constexpr int PROJ = EPI_BIAS | EPI_RES1 | EPI_RES2;                     // x = v M^T + b + pos_emb + x
        // bf16 activations: operand tiles come through the TMA engine (thread-loader kernel as fall-back when
        // the tensor map cannot be built: unaligned views)
#define TMA_CASE(BN_, KP_, EPI_) \
        if (!ln && p.K == KP_ && p.Np % BN_ == 0 && epi == (EPI_) && launch_tma_t<BN_, KP_, (EPI_)>(cx, p, name)) return true;
        TMA_CASE(32, 32, PROJ) TMA_CASE(64, 64, PROJ) TMA_CASE(128, 128, PROJ)
#undef TMA_CASE
        PW_CASE(32, 32, false, PROJ) PW_CASE(64, 64, false, PROJ) PW_CASE(128, 128, false, PROJ)
    } else {
        constexpr int FFN0 = EPI_GELU | EPI_OUTBF16, UP = EPI_BIAS | EPI_CONVT;
        PW_CASE(256, 64, true, FFN0) PW_CASE(256, 128, true, FFN0)
        // q | k | v: fp32 activations through the TMA engine, tf32 tensor cores (thread-loader kernel as fall-back)
#define TMA32_CASE(BN_, KP_, EPI_) \
        if (!ln && p.W32 && p.K == KP_ && p.Np % BN_ == 0 && epi == (EPI_) && launch_tma32_t<BN_, KP_, (EPI_)>(cx, p, name)) return true;
        TMA32_CASE(96, 32, EPI_OUTBF16) TMA32_CASE(192, 64, EPI_OUTBF16) TMA32_CASE(128, 128, EPI_OUTBF16)
#undef TMA32_CASE
        PW_CASE(96, 32, false, EPI_OUTBF16) PW_CASE(192, 64, false, EPI_OUTBF16) PW_CASE(192, 128, false, EPI_OUTBF16)   // q | k | v
        PW_CASE(256, 128, false, UP) PW_CASE(128, 64, false, UP)                 // ConvTranspose2d(2, 2)
        PW_CASE(64, 128, false, 0) PW_CASE(32, 64, false, 0)                     // 1x1 fusion of cat([up, skip])
    }
#undef PW_CASE
    return false;
}

template <bool A_BF16, int MODE>
static void launch_gemm(Ctx &cx, const GemmP &p, const char *name) {
    if constexpr (MODE == MODE_PW) {
        if (launch_pw<A_BF16>(cx, p, name)) return;
    }
    if (p.ln_g || p.zero_ptr) { cx.unsupported = 1; return; }      // the generic kernel has no fused LayerNorm / clear
    // one CTA covers as many output channels as one tcgen05.mma can (N <= 256): the A tile is read once
    if (p.Np % 256 == 0) launch_gemm_t<256, A_BF16, MODE>(cx, p, name);
    else if (p.Np % 192 == 0) launch_gemm_t<192, A_BF16, MODE>(cx, p, name);
    else if (p.Np % 128 == 0) launch_gemm_t<128, A_BF16, MODE>(cx, p, name);
    else if (p.Np % 96 == 0) launch_gemm_t<96, A_BF16, MODE>(cx, p, name);
    else if (p.Np % 64 == 0) launch_gemm_t<64, A_BF16, MODE>(cx, p, name);
    else launch_gemm_t<32, A_BF16, MODE>(cx, p, name);
}

static GemmP gemm_defaults() {
    GemmP p{};
    p.out_mode = OUT_ROWS;
    return p;
}

// 3x3 conv on [B, H, W, 32]: the row-streaming kernel when the map is a whole number of 128-column strips,
// the K-chunked implicit GEMM otherwise
static void launch_conv3(Ctx &cx, const GemmP &p, const char *name) {
    const int H = p.Hi, W = p.Wi;
    if (W % BM != 0 || H < 2) {
        launch_gemm<false, MODE_C3>(cx, p, name);
        return;
    }
    // rows per CTA: ~2 CTAs per SM over the batch, at least 8 rows (2 halo rows are re-read per segment)
    const int strips = W / BM;
    int segs = std::max(1, (2 * sm_count()) / std::max(1, strips * cx.B));
    int seg_rows = std::max(8, (H + segs - 1) / segs);
    segs = (H + seg_rows - 1) / seg_rows;
    const dim3 grid(strips, segs, cx.B);
    const int epi = tc::epi_of(p);
    AVB_TIMED(name, cx.st);
#define C3_CASE(EPI_) \
    if (epi == (EPI_) && p.out_mode != OUT_CROP) { \
        static SmemOptIn opt_in; \
        opt_in.ensure(tc::conv3_stream_kernel<(EPI_)>, tc::C3_SMEM); \
        cudaLaunchConfig_t cfg = {}; cfg.gridDim = grid; cfg.blockDim = dim3(GEMM_THREADS); cfg.dynamicSmemBytes = tc::C3_SMEM; cfg.stream = cx.st; \
        cudaLaunchAttribute attr[1]; attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization; attr[0].val.programmaticStreamSerializationAllowed = 1; \
        cfg.attrs = attr; cfg.numAttrs = 1; \
        cudaLaunchKernelEx(&cfg, tc::conv3_stream_kernel<(EPI_)>, p, seg_rows); \
        return; \
    }
    C3_CASE(0) C3_CASE(tc::EPI_RES1)
#undef C3_CASE
    {   // conv_out: cropped store (runtime epilogue flags)
        static SmemOptIn opt_in;
        opt_in.ensure(tc::conv3_stream_kernel<tc::EPI_RUNTIME>, tc::C3_SMEM);
        cudaLaunchConfig_t cfg = {}; cfg.gridDim = grid; cfg.blockDim = dim3(GEMM_THREADS); cfg.dynamicSmemBytes = tc::C3_SMEM; cfg.stream = cx.st;
        cudaLaunchAttribute attr[1]; attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization; attr[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = attr; cfg.numAttrs = 1;
        cudaLaunchKernelEx(&cfg, tc::conv3_stream_kernel<tc::EPI_RUNTIME>, p, seg_rows);
    }
}

static void conv3x3(Ctx &cx, const float *in, const bf16 *w, float *out, const float *res, int H, int W) {
    GemmP p = gemm_defaults();
    p.A1 = in; p.lda1 = 32; p.K1 = p.K = 288; p.W = w; p.Np = 32; p.rows = H * W;
    p.Hi = p.Ho = H; p.Wi = p.Wo = W; p.Cpin = 32;
    p.res1 = res; p.ldr1 = 32; p.out = out; p.ldo = 32;
    launch_conv3(cx, p, "k4_conv3x3");
}

static void dwconv(Ctx &cx, const bf16 *in, int ldi, bf16 *out, int ldo, const float *w, int H, int W, int Cp, int gelu_out, const char *name) {
    // rows per thread: long enough to amortise the 2 halo rows, short enough to fill the machine
    const long long items = (long long)cx.B * H * W * (Cp / DW_CPT);
    const int seg = (int)std::max<long long>(4, std::min<long long>(32, items / ((long long)sm_count() * 1024)));
    DwP p{in, ldi, out, ldo, w, cx.B, H, W, Cp, gelu_out, seg};
    const long long total = (long long)cx.B * ((H + seg - 1) / seg) * W * (Cp / DW_CPT);
    AVB_TIMED(name, cx.st);
    if (Cp % DP_CB == 0 && (ldi & 7) == 0 && (reinterpret_cast<uintptr_t>(in) & 15) == 0) {
        launch_pdl(dwconv_tile_kernel, dim3((W + DP_TX - 1) / DP_TX, (H + DP_TY - 1) / DP_TY, cx.B * (Cp / DP_CB)), dim3(256), 0, cx.st, p);
        return;
    }
    launch_pdl(dwconv_kernel<DW_CPT>, dim3((unsigned)((total + 127) / 128)), dim3(128), 0, cx.st, p);
}

// FeedForward behind its PreNorm in one kernel per 128 hidden channels: x = xin + W4 GELU(dw(GELU(W0 LN(xin))))
template <int CP>
static void ffn_fused_launch(Ctx &cx, const MsabW &m, const float *xin, float *x, int H, int W) {
    typedef tc::FfnCfg<CP> Cfg;
    static SmemOptIn opt_in;              // per instantiation, per device
    opt_in.ensure(tc::ffn_fused_kernel<CP>, Cfg::SMEM);
    // strips of <= 126 output columns (128 with the x halo = one MMA tile), row segments so that one CTA per SM is busy
    const int strips = (W + 125) / 126, strip_w = (W + strips - 1) / strips;
    int segs = std::max(1, sm_count() / std::max(1, strips * cx.B));
    const int seg_rows = std::max(std::min(H, 4), (H + segs - 1) / segs);
    segs = (H + seg_rows - 1) / seg_rows;
    if ((long long)cx.B * H * W * CP >= (1LL << 31)) { cx.unsupported = 1; return; }      // 32-bit element offsets inside the kernel
    for (int ck = 0; ck < m.Hp / tc::FF_HC; ++ck) {
        tc::FfnP p{xin, ck == 0 ? xin : x, x, m.ffn_blob + (size_t)ck * Cfg::BLOB, m.ffn_dw + ck * tc::FF_HC, m.ln_g, m.ln_b, m.Hp, m.c, H, W, strip_w, seg_rows};
        AVB_TIMED("k4_ffn_fused", cx.st);
        launch_pdl(tc::ffn_fused_kernel<CP>, dim3(strips, segs, cx.B), dim3(tc::FF_THREADS), Cfg::SMEM, cx.st, p);
    }
}

// MSAB with num_blocks = 1 (MST_Plus_Plus.py:160-186), in place on x (fp32 [B*rows, Cp]).
static void msab(Ctx &cx, const MsabW &m, float *x, int H, int W, Workspace &ws) {
    const int rows = H * W, Cp = m.Cp, Hp = m.Hp;
    // q | k | v
    {
        GemmP p = gemm_defaults();
        p.A1 = x; p.lda1 = Cp; p.K1 = p.K = Cp; p.W = m.wqkv; p.W32 = m.wqkv32; p.Np = 3 * Cp; p.rows = rows;
        p.out = ws.qkv; p.ldo = 3 * Cp; p.out_bf16 = 1;
        // tickets | statistics (int64 entries, accumulated with atomics): one contiguous clear
        p.zero_ptr = reinterpret_cast<float *>(ws.tickets);
        p.zero_n = (int)(reinterpret_cast<float *>(ws.stats) - reinterpret_cast<float *>(ws.tickets)) + 2 * cx.B * m.heads * 1024;
        launch_gemm<false, MODE_PW>(cx, p, "k4_gemm_qkv");
    }
    {
        // statistics (+ softmax / M by the last CTA of every head) and the positional embedding in one launch
        AttnSideP p{};
        p.st = AttnStatP{ws.qkv, ws.stats, rows, Cp, m.heads, 0};
#ifndef AVB_STATS_PER_SM
#define AVB_STATS_PER_SM 2     // statistics CTAs per SM and head group (measured, forward: 1 -> 3.12 ms, 2 -> 2.98, 3 -> 2.97, 4 -> 3.00)
#endif
        int ctas = std::max(1, std::min((rows + 255) / 256, sm_count() * AVB_STATS_PER_SM / std::max(1, m.heads)));     // geometry only: batch invariant
        p.st.px_per_cta = ((rows + ctas - 1) / ctas + 127) / 128 * 128;
        ctas = (rows + p.st.px_per_cta - 1) / p.st.px_per_cta;
        p.fin = AttnFinP{ws.stats, m.rescale, m.wproj_f32, ws.M, m.c, Cp, m.heads};
        p.dp = DwPosP{ws.qkv + 2 * Cp, 3 * Cp, ws.p2, Cp, m.pos0, m.pos2, cx.B, H, W, Cp};
        p.tickets = ws.tickets;
        p.ctasA = ctas; p.nA = ctas * m.heads * cx.B;
        p.gx = (W + DP_TX - 1) / DP_TX; p.gy = (H + DP_TY - 1) / DP_TY;
        const long long total = (long long)p.nA + (long long)p.gx * p.gy * cx.B * (Cp / DP_CB);
        AVB_TIMED("k4_attn_side", cx.st);
        launch_pdl(attn_side_kernel, dim3((unsigned)total), dim3(128), 0, cx.st, p);
    }
    // the full-resolution level (Cp == 32) runs its feed-forward block as one fused kernel, the coarser levels as three.
    // The fused kernel reads halo rows of its input while neighbouring CTAs write the output: the attention block then
    // leaves its result in ws.xt and the feed-forward block brings it back to x
    const bool ffn_fused = Cp == 32;
    // x = v M^T + b + pos + x
    {
        GemmP p = gemm_defaults();
        p.A1 = ws.qkv + 2 * Cp; p.lda1 = 3 * Cp; p.K1 = p.K = Cp; p.W = ws.M; p.w_bstride = (long long)Cp * Cp; p.Np = Cp; p.rows = rows;
        p.bias = m.bproj; p.res1 = x; p.ldr1 = Cp; p.res2 = ws.p2; p.ldr2 = Cp; p.out = ffn_fused ? ws.xt : x; p.ldo = Cp;
        launch_gemm<true, MODE_PW>(cx, p, "k4_gemm_attn_proj");
    }
    if (ffn_fused) {
        ffn_fused_launch<32>(cx, m, ws.xt, x, H, W);
        return;
    }
    // FFN: x = W4 GELU(dw(GELU(W0 LN(x)))) + x; the LayerNorm runs inside the FFN-in GEMM's loader
    {
        GemmP p = gemm_defaults();
        p.A1 = x; p.lda1 = Cp; p.K1 = p.K = Cp; p.W = m.ffn0; p.Np = Hp; p.rows = rows;
        p.ln_g = m.ln_g; p.ln_b = m.ln_b; p.ln_c = m.c;
        p.gelu = 1; p.out = ws.hid1; p.ldo = Hp; p.out_bf16 = 1;
        launch_gemm<false, MODE_PW>(cx, p, "k4_gemm_ln_ffn0");
    }
    dwconv(cx, ws.hid1, Hp, ws.hid2, Hp, m.ffn_dw, H, W, Hp, 1, "k4_dw_ffn");
    {
        GemmP p = gemm_defaults();
        p.A1 = ws.hid2; p.lda1 = Hp; p.K1 = p.K = Hp; p.W = m.ffn4; p.Np = Cp; p.rows = rows;
        p.res1 = x; p.ldr1 = Cp; p.out = x; p.ldo = Cp;
        launch_gemm<true, MODE_PW>(cx, p, "k4_gemm_ffn4");
    }
}

// MST body (MST_Plus_Plus.py:240-268): in -> out (both fp32 [B, H, W, 32])
static void mst_body(Ctx &cx, const BodyW &Bw, const float *in, float *out, int H, int W, Workspace &ws) {
    conv3x3(cx, in, Bw.embedding, ws.f0, nullptr, H, W);
    float *lvl[3] = {ws.f0, ws.f1, ws.f2};
    int h = H, w = W, c = NF;
    for (int i = 0; i < 2; ++i) {
        msab(cx, Bw.enc[i], lvl[i], h, w, ws);
        GemmP p = gemm_defaults();       // Conv2d(c, 2c, 4, 2, 1)
        p.A1 = lvl[i]; p.lda1 = pad32(c); p.Cpin = pad32(c); p.K1 = p.K = 16 * pad32(c); p.W = Bw.down[i]; p.Np = pad32(2 * c);
        p.Hi = h; p.Wi = w; p.Ho = h / 2; p.Wo = w / 2; p.rows = (h / 2) * (w / 2);
        p.out = lvl[i + 1]; p.ldo = pad32(2 * c);
        launch_gemm<false, MODE_C4S2>(cx, p, "k4_conv4x4s2");
        h /= 2; w /= 2; c *= 2;
    }
    msab(cx, Bw.bott, ws.f2, h, w, ws);
    float *cur = ws.f2;
    float *ups[2] = {ws.u1, ws.u0}, *decs[2] = {ws.d1, ws.d0}, *skips[2] = {ws.f1, ws.f0};
    for (int i = 0; i < 2; ++i) {
        const int co = c / 2, Cpi = pad32(c), Cpo = pad32(co);
        {   // ConvTranspose2d(c, c/2, 2, 2) + bias
            GemmP p = gemm_defaults();
            p.A1 = cur; p.lda1 = Cpi; p.K1 = p.K = Cpi; p.W = Bw.up[i]; p.Np = 4 * Cpo; p.rows = h * w;
            p.Ho = h; p.Wo = w; p.bias = Bw.up_bias[i]; p.out = ups[i]; p.ldo = Cpo; p.out_mode = OUT_CONVT; p.Cpo = Cpo;
            launch_gemm<false, MODE_PW>(cx, p, "k4_convT2x2");
        }
        h *= 2; w *= 2;
        {   // 1x1 fusion of cat([up, skip])
            GemmP p = gemm_defaults();
            p.A1 = ups[i]; p.lda1 = Cpo; p.A2 = skips[i]; p.lda2 = Cpo; p.K1 = Cpo; p.K = 2 * Cpo; p.W = Bw.fuse[i]; p.Np = Cpo; p.rows = h * w;
            p.out = decs[i]; p.ldo = Cpo;
            launch_gemm<false, MODE_PW>(cx, p, "k4_gemm_fuse");
        }
        msab(cx, Bw.dec[i], decs[i], h, w, ws);
        cur = decs[i];
        c = co;
    }
    conv3x3(cx, cur, Bw.mapping, out, in, H, W);      // mapping(fea) + x
}

}  // namespace k4
}  // namespace avb

using namespace avb;
using namespace avb::k4;

extern "C" int avb_mstpp_create(const float *params_host, int64_t count, void **handle) {
    AVB_REQUIRE(params_host && handle, "null pointer");
    if (count != N_PARAMS) {
        set_error("avb_mstpp_create: expected %lld float32 parameters (MST_Plus_Plus state_dict order), got %lld",
                  (long long)N_PARAMS, (long long)count);
        return AVB_E_ARG;
    }
    Model *M = new Model();
    Packer pk;
    pk.host.reserve(8u << 20);
    if (!pack_model(pk, *M, params_host, count)) {
        delete M;
        set_error("avb_mstpp_create: parameter blob does not match the MST++ architecture");
        return AVB_E_ARG;
    }
    cudaError_t e = cudaGetDevice(&M->device);
    if (e == cudaSuccess) e = cudaMalloc(&M->blob, pk.host.size());
    if (e == cudaSuccess) e = cudaMemcpy(M->blob, pk.host.data(), pk.host.size(), cudaMemcpyHostToDevice);
    if (e != cudaSuccess) {
        delete M;
        return cuda_fail(e, "avb_mstpp_create upload");
    }
    for (auto &f : pk.fixes) *f.slot = static_cast<uint8_t *>(M->blob) + f.off;
    *handle = M;
    return AVB_OK;
}

extern "C" int avb_mstpp_destroy(void *handle) {
    if (!handle) return AVB_OK;
    Model *M = static_cast<Model *>(handle);
    cudaFree(M->blob);
    delete M;
    return AVB_OK;
}

static void padded_geometry(int H, int W, int multiple, int centred, int &Hp, int &Wp, int &top, int &left) {
    const int ph = (multiple - H % multiple) % multiple, pw = (multiple - W % multiple) % multiple;
    Hp = H + ph; Wp = W + pw;
    top = centred ? ph / 2 : 0;
    left = centred ? pw / 2 : 0;
}

extern "C" int64_t avb_mstpp_workspace_bytes(int n, int H, int W, int pad_multiple, int centred) {
    if (n <= 0 || H <= 1 || W <= 1 || pad_multiple <= 0 || pad_multiple % 8) return 0;
    int Hp, Wp, top, left;
    padded_geometry(H, W, pad_multiple, centred, Hp, Wp, top, left);
    return (int64_t)carve(nullptr, nullptr, n, Hp, Wp);
}

extern "C" int avb_mstpp_forward_bands(void *handle, const void *in, int in_is_u8, float *out, float *bands_out,
                                       const float *band_weights_dev, int n_bands, int n, int H, int W,
                                       int pad_multiple, int centred, void *workspace_dev, avb_stream_t stream);

extern "C" int avb_mstpp_forward(void *handle, const void *in, int in_is_u8, float *out, int n, int H, int W,
                                 int pad_multiple, int centred, void *workspace_dev, avb_stream_t stream) {
    AVB_REQUIRE(out, "null pointer");
    return avb_mstpp_forward_bands(handle, in, in_is_u8, out, nullptr, nullptr, 0, n, H, W, pad_multiple, centred, workspace_dev, stream);
}

extern "C" int avb_mstpp_forward_bands(void *handle, const void *in, int in_is_u8, float *out, float *bands_out,
                                       const float *band_weights_dev, int n_bands, int n, int H, int W,
                                       int pad_multiple, int centred, void *workspace_dev, avb_stream_t stream) {
    AVB_REQUIRE(handle && in && workspace_dev && (out || bands_out), "null pointer");
    AVB_REQUIRE((bands_out == nullptr) == (n_bands == 0) && (bands_out == nullptr || band_weights_dev) && n_bands >= 0 && n_bands <= 64,
                "bands_out, band_weights_dev and n_bands (1..64) go together");
    AVB_REQUIRE(n > 0 && n <= 65535 && H > 1 && W > 1, "bad geometry");
    AVB_REQUIRE(pad_multiple > 0 && pad_multiple % 8 == 0, "pad_multiple must be a positive multiple of 8");
    Model *M = static_cast<Model *>(handle);
    int cur_dev = -1;
    AVB_CUDA_OK(cudaGetDevice(&cur_dev));
    if (cur_dev != M->device) {            // the weights live on the device the model was created on
        set_error("avb_mstpp_forward: model was created on device %d, current device is %d", M->device, cur_dev);
        return AVB_E_ARG;
    }
    int Hp, Wp, top, left;
    padded_geometry(H, W, pad_multiple, centred, Hp, Wp, top, left);
    AVB_REQUIRE(Hp - H < H && Wp - W < W, "frame too small for reflect padding");
    Workspace ws{};
    carve(&ws, static_cast<uint8_t *>(workspace_dev), n, Hp, Wp);
    Ctx cx{static_cast<cudaStream_t>(stream), n};
    {
        ConvInP p{in, in_is_u8, ws.x0, M->conv_in, n, H, W, Hp, Wp, top, left};
        const long long npx = (long long)n * Hp * Wp;
        AVB_TIMED("k4_conv_in", cx.st);
        launch_pdl(conv_in_kernel, dim3((unsigned)((npx + 127) / 128)), dim3(128), 0, cx.st, p);
    }
    const float *hin = ws.x0;
    float *pp[2] = {ws.hA, ws.hB};
    for (int s = 0; s < 3; ++s) {
        mst_body(cx, M->body[s], hin, pp[s & 1], Hp, Wp, ws);
        hin = pp[s & 1];
    }
    {   // conv_out(h) + conv_in(x), cropped to the input size, NHWC with 31 packed channels
        GemmP p = gemm_defaults();
        p.A1 = hin; p.lda1 = 32; p.K1 = p.K = 288; p.W = M->conv_out; p.Np = 32; p.rows = Hp * Wp;
        p.Hi = p.Ho = Hp; p.Wi = p.Wo = Wp; p.Cpin = 32;
        p.res1 = ws.x0; p.ldr1 = 32; p.out = out; p.out_mode = OUT_CROP; p.Hreal = H; p.Wreal = W; p.crop_top = top; p.crop_left = left;
        if (bands_out) {
            AVB_CUDA_OK(cudaMemsetAsync(bands_out, 0, sizeof(float) * (size_t)n * H * W * n_bands, cx.st));
            p.band_w = band_weights_dev; p.bands_out = bands_out; p.n_bands = n_bands;
        }
        launch_conv3(cx, p, "k4_conv3x3");
    }
    AVB_REQUIRE(!cx.unsupported, "layer shape without a kernel");
    AVB_CUDA_OK(cudaGetLastError());
    return AVB_OK;
}

extern "C" int avb_safe_norm_f32(const float *in_dev, float *out_dev, int64_t npx, int stride, int n_maps,
                                 void *scratch_dev, avb_stream_t stream) {
    AVB_REQUIRE(in_dev && out_dev && scratch_dev, "null pointer");
    AVB_REQUIRE(npx > 0 && n_maps > 0 && n_maps <= 65535 && stride >= n_maps, "bad map geometry");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    uint32_t *mm = static_cast<uint32_t *>(scratch_dev);
    AVB_CUDA_OK(cudaMemsetAsync(mm, 0xff, sizeof(uint32_t) * n_maps, st));            // minima: +inf in ordered form
    AVB_CUDA_OK(cudaMemsetAsync(mm + n_maps, 0x00, sizeof(uint32_t) * n_maps, st));   // maxima: -inf in ordered form
    const int bx = (int)std::min<long long>((npx + 255) / 256, (long long)sm_count() * 8);
    {
        AVB_TIMED("safe_norm_minmax", st);
        minmax_kernel<<<dim3(bx, n_maps), 256, 0, st>>>(in_dev, npx, stride, n_maps, mm);
    }
    {
        AVB_TIMED("safe_norm", st);
        safe_norm_kernel<<<dim3(bx, n_maps), 256, 0, st>>>(in_dev, out_dev, npx, stride, n_maps, mm);
    }
    AVB_CUDA_OK(cudaGetLastError());
    return AVB_OK;
}

extern "C" int avb_band_project_f32(const float *cube_dev, const float *weights_dev, float *out_dev,
                                    int64_t npx, int n_bands, int n_receptors, avb_stream_t stream) {
    AVB_REQUIRE(cube_dev && weights_dev && out_dev, "null pointer");
    AVB_REQUIRE(npx > 0 && n_bands > 0 && n_receptors > 0 && n_bands * n_receptors <= 8192, "bad projection geometry");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const long long total = npx * n_receptors;
    const int blocks = (int)std::min<long long>((total + 255) / 256, (long long)sm_count() * 16);
    AVB_TIMED("k4_band_project", st);
    band_project_kernel<<<blocks, 256, sizeof(float) * n_bands * n_receptors, st>>>(cube_dev, weights_dev, out_dev, npx, n_bands, n_receptors);
    AVB_CUDA_OK(cudaGetLastError());
    return AVB_OK;
}
