// K11 -- packs n encoded frames (K8's slots) into contiguous AVI '00dc' chunks, the records of a Motion-JPEG AVI's
// 'movi' list (animal_vision_b200/renderers/mjpeg.py writes them to the file as they are).  A record is the fourcc, a
// little-endian u32 size, the JPEG, then zero bytes up to a multiple of 4; the size counts the padding, as OpenCV's
// AVI writer stores it.  A chunk of frames thus becomes one region that crosses to the host in one copy.
//
//   mjpeg_pack  grid (CTAs per frame, n): every CTA sums the padded sizes of the frames before its own (n is a chunk of
//               frames, a few dozen at most), so no scan launch precedes the copy.  The copy writes whole 32-bit words
//               of the record: each is two aligned source words joined by a funnel shift (the slots of K8 start at any
//               byte), 16-byte stores where the destination is 16-byte aligned.
#include "avb_common.cuh"

namespace {

constexpr int PACK_THREADS = 256;

__device__ __forceinline__ int64_t slot_len(const int64_t *lengths, int f, int64_t slot) {
    return min(max(lengths[f], (int64_t)0), slot);
}

__device__ __forceinline__ int64_t record_bytes(int64_t len) { return 8 + ((len + 3) & ~(int64_t)3); }

// word k of the padded JPEG that starts at src and is len bytes long: bytes src[4k, 4k + 4), zero past len.  Reads only
// aligned words that hold at least one byte of the JPEG.
__device__ __forceinline__ uint32_t src_word(const uint8_t *src, int64_t len, int64_t k) {
    const uintptr_t p = (uintptr_t)src + 4 * k;
    const int s = (int)(p & 3);
    const uint32_t *a = reinterpret_cast<const uint32_t *>(p - s);
    uint32_t v = __ldg(a);
    if (s) v = __funnelshift_r(v, 4 * k + 4 - s < len ? __ldg(a + 1) : 0u, 8 * s);
    const int64_t valid = len - 4 * k;
    if (valid < 4) v &= (1u << (8 * valid)) - 1u;
    return v;
}

__global__ void __launch_bounds__(PACK_THREADS) mjpeg_pack_kernel(const uint8_t *__restrict__ slots, int64_t slot,
                                                                  const int64_t *__restrict__ lengths, int n,
                                                                  uint8_t *__restrict__ out, int64_t *offsets) {
    __shared__ int64_t s_off;
    const int f = blockIdx.y;
    if (threadIdx.x < 32) {                       // offset of this frame's record: the padded records before it
        int64_t acc = 0;
        for (int i = threadIdx.x; i < f; i += 32) acc += record_bytes(slot_len(lengths, i, slot));
#pragma unroll
        for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        if (threadIdx.x == 0) s_off = acc;
    }
    __syncthreads();
    const int64_t off = s_off, len = slot_len(lengths, f, slot), words = (len + 3) >> 2;
    uint8_t *rec = out + off;
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        reinterpret_cast<uint32_t *>(rec)[0] = 0x63643030u;          // "00dc"
        reinterpret_cast<uint32_t *>(rec)[1] = (uint32_t)(4 * words);
        offsets[f] = off;
        if (f == n - 1) offsets[n] = off + 8 + 4 * words;
    }
    const uint8_t *src = slots + (int64_t)f * slot;
    uint32_t *dst = reinterpret_cast<uint32_t *>(rec + 8);
    // words [0, head) and [head + 4 * units, words) one at a time, the 16-byte aligned units between them whole
    const int64_t head = min((int64_t)((16 - ((uintptr_t)dst & 15)) & 15) >> 2, words);
    const int64_t units = (words - head) >> 2, tail0 = head + 4 * units;
    const int64_t t0 = (int64_t)blockIdx.x * PACK_THREADS + threadIdx.x, stride = (int64_t)gridDim.x * PACK_THREADS;
    for (int64_t u = t0; u < units; u += stride) {
        const int64_t k = head + 4 * u;
        uint4 v;
        v.x = src_word(src, len, k);
        v.y = src_word(src, len, k + 1);
        v.z = src_word(src, len, k + 2);
        v.w = src_word(src, len, k + 3);
        reinterpret_cast<uint4 *>(dst + k)[0] = v;
    }
    if (t0 < head) dst[t0] = src_word(src, len, t0);
    if (t0 < words - tail0) dst[tail0 + t0] = src_word(src, len, tail0 + t0);
}

}  // namespace

extern "C" int avb_mjpeg_pack_u8(const uint8_t *slots, int64_t slot_stride, const int64_t *lengths_dev, int n,
                                 uint8_t *out, int64_t *out_offsets_dev, avb_stream_t stream) {
    AVB_REQUIRE(slots && lengths_dev && out && out_offsets_dev, "null pointer");
    AVB_REQUIRE(n >= 1 && n <= 65535, "n must lie in [1, 65535]");
    AVB_REQUIRE(slot_stride >= 1, "slot_stride must be positive");
    AVB_REQUIRE(((uintptr_t)slots & 3) == 0 && ((uintptr_t)out & 15) == 0, "slots must be 4-byte, out 16-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    const int per_frame = (avb::sm_count() * 4 + n - 1) / n;
    {
        AVB_TIMED("mjpeg_pack", st);
        mjpeg_pack_kernel<<<dim3(per_frame, n), PACK_THREADS, 0, st>>>(slots, slot_stride, lengths_dev, n, out,
                                                                       out_offsets_dev);
    }
    AVB_CUDA_OK(cudaGetLastError());
    return AVB_OK;
}
