// Shared host/device helpers for libavb200 (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <stdio.h>

#include <atomic>

#include "../../include/avb200.h"

namespace avb {

// ---------------------------------------------------------------- errors
void set_error(const char *fmt, ...);
int cuda_fail(cudaError_t e, const char *what);

#define AVB_CUDA_OK(expr)                                     \
    do {                                                      \
        cudaError_t _e = (expr);                              \
        if (_e != cudaSuccess) return avb::cuda_fail(_e, #expr); \
    } while (0)

#define AVB_REQUIRE(cond, msg)                  \
    do {                                        \
        if (!(cond)) {                          \
            avb::set_error("%s: %s", __func__, msg); \
            return AVB_E_ARG;                   \
        }                                       \
    } while (0)

int sm_count();  // multiprocessors of the current device (cached)

// cudaFuncAttributeMaxDynamicSharedMemorySize is a PER-DEVICE attribute of a kernel: remember, per call
// site, on which devices it has been set (a process may drive several GPUs, one Engine per device).
struct SmemOptIn {
    std::atomic<uint64_t> done{0};
    template <class K>
    cudaError_t ensure(K kern, int bytes) {
        int dev = 0;
        cudaError_t e = cudaGetDevice(&dev);
        if (e != cudaSuccess) return e;
        const bool tracked = dev >= 0 && dev < 64;
        if (tracked && ((done.load(std::memory_order_acquire) >> dev) & 1ull)) return cudaSuccess;
        e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
        if (e == cudaSuccess && tracked) done.fetch_or(1ull << dev, std::memory_order_release);   // idempotent: a race only repeats it
        return e;
    }
};

// ---------------------------------------------------------------- numpy.percentile(float32 data, python-float q)
// NumPy divides q by float32(100) and keeps the virtual index (n-1)*q in FLOAT32 (numpy/lib/_function_base_impl.py:
// percentile -> _quantile -> _lerp); the two neighbouring order statistics are blended in float32, from the upper
// one when the weight is >= 0.5.  Restated exactly (3000/3000 random cases bit-equal in tools/probe notes, DESIGN.md).
struct PctIndex {
    long long k_lo, k_hi;
    float gamma;
};
inline PctIndex numpy_percentile_index(double q, long long n) {
    const float qq = (float)q / 100.0f;
    const float vi = (float)(n - 1) * qq;
    PctIndex r;
    r.k_lo = (long long)floorf(vi);
    if (r.k_lo > n - 1) r.k_lo = n - 1;
    if (r.k_lo < 0) r.k_lo = 0;
    r.k_hi = r.k_lo + 1 < n ? r.k_lo + 1 : r.k_lo;
    r.gamma = vi - (float)r.k_lo;
    if (r.gamma < 0.f) r.gamma = 0.f;
    return r;
}
__device__ __forceinline__ float numpy_lerp(float a, float b, float g) {
    const float d = __fsub_rn(b, a);
    return g >= 0.5f ? __fsub_rn(b, __fmul_rn(d, __fsub_rn(1.0f, g))) : __fadd_rn(a, __fmul_rn(d, g));
}

// ---------------------------------------------------------------- per-kernel timing (bench only)
// Between avb_profile_begin() and avb_profile_end() every kernel launched by the library on the
// calling thread is bracketed by a pair of CUDA events on its own stream.  Off by default.
bool profiling_on();
void profile_mark(const char *name, cudaStream_t st, bool begin);

struct LaunchScope {
    const char *name;
    cudaStream_t st;
    bool on;
    LaunchScope(const char *n, cudaStream_t s) : name(n), st(s), on(profiling_on()) {
        if (on) profile_mark(name, st, true);
    }
    ~LaunchScope() {
        if (on) profile_mark(name, st, false);
    }
};
#define AVB_TIMED(name, st) avb::LaunchScope _avb_scope_##__LINE__(name, st)

// ---------------------------------------------------------------- frame addressing
struct FrameIO {
    const uint8_t *in;
    uint8_t *out;
    int64_t in_fs, in_rs, out_fs, out_rs;  // byte strides
    int n, H, W;
};

struct Mat3 {
    float m[9];
};

// ---------------------------------------------------------------- encode table
// Layout of the table built by avb_build_encode_table:
//   [0] key_min   (float bits >> shift of the first bucket)
//   [1] shift     (23 - mantissa bits kept)
//   [2] n_buckets
//   [3] reserved
//   [4 .. 4+n_buckets) entries: (threshold_low_bits << 8) | byte_at_bucket_start
// A bucket is the set of floats sharing (bits >> shift); it contains at most one quantisation
// threshold, stored as its low `shift` bits (or 1<<shift when the bucket has none).
constexpr int ENC_HEADER = 4;

struct EncTable {            // view over shared memory
    const uint32_t *e;       // entries
    uint32_t lo_bits;        // key_min << shift : everything below encodes to byte 0
    uint32_t shift;
    uint32_t mask;
};

__device__ __forceinline__ EncTable enc_view(const uint32_t *smem_table) {
    EncTable t;
    t.shift = smem_table[1];
    t.lo_bits = smem_table[0] << t.shift;
    t.mask = (1u << t.shift) - 1u;
    t.e = smem_table + ENC_HEADER;
    return t;
}

// clip(x,0,1) -> OETF -> *255+0.5 -> truncate, as one table lookup.  NaN encodes to 0.
__device__ __forceinline__ uint32_t encode_u8(const EncTable &t, float x) {
    uint32_t b = __float_as_uint(__saturatef(x));
    b = max(b, t.lo_bits);
    uint32_t ent = t.e[(b - t.lo_bits) >> t.shift];
    return (ent & 0xffu) + (((b & t.mask) >= (ent >> 8)) ? 1u : 0u);
}

__device__ __forceinline__ int reflect101(int i, int n) {
    // cv::borderInterpolate(BORDER_REFLECT_101); loops only for overshoots beyond one period
    if (n == 1) return 0;
    while ((unsigned)i >= (unsigned)n) i = (i < 0) ? -i : 2 * n - 2 - i;
    return i;
}

// cooperative copy of a small global table into shared memory
__device__ __forceinline__ void copy_to_smem(uint32_t *dst, const uint32_t *src, int n) {
    for (int i = threadIdx.x; i < n; i += blockDim.x) dst[i] = __ldg(src + i);
}

}  // namespace avb
