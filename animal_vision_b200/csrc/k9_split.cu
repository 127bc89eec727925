// K9: the labelled split-compare frame of make_split_frame (reference renderers/video.py:198-245) for a batch.
//
// Columns [0, W/2) come from `left`, [W/2, W) from `right`, column W/2 is set to 255 when the seam is on, and in the
// label band (rows [0, band_rows)) every byte b of a pixel of class c becomes lut[c][b].  The tables are the corner
// labels of draw_split_labels as a per-pixel byte map (animal_vision_b200/tables.py split_label_stencil): the label
// drawing reads no neighbouring pixel and treats the three channels alike, so a 256-entry table per pixel position
// states it exactly, and the device frame has the bytes of the host drawing.
//
// A streaming kernel: 3 B/px in, 3 B/px out; the class map ([band_rows, W] uint16) and the tables ([classes, 256]) are
// a few hundred kB and stay in L2.  One CTA covers CHUNKS_PER_CTA V-byte chunks of one output row, each thread two of
// them (both loads issued before the stores).  V = 16 when every base pointer and stride allows 16-byte accesses,
// else 4, else 1.  Outside the band a chunk is one load and one store; only the chunk that holds the left/right
// boundary or the seam, and a row's partial last chunk, touch single bytes.
#include "avb_common.cuh"

namespace {

constexpr int THREADS = 64;
constexpr int UNROLL = 2;
constexpr int CHUNKS_PER_CTA = THREADS * UNROLL;
constexpr int MIN_CTAS = 16;     // 1024 threads per SM: 64 registers, no spills (80 unbounded)

struct SplitArgs {
    const uint8_t *left, *right;
    uint8_t *out;
    int64_t lfs, lrs, rfs, rrs, ofs, ors;
    int n, H, W;
    int row_bytes;   // 3W
    int split;       // first byte of the right half, 3 * (W / 2)
    int seam;        // write 255 to bytes [split, split + 3)
    int band_rows;
    const uint16_t *cls;   // [band_rows, W]
    const uint8_t *lut;    // [classes, 256]
};

template <int V>
struct Vec;
template <>
struct Vec<16> {
    using T = uint4;
};
template <>
struct Vec<4> {
    using T = uint32_t;
};
template <>
struct Vec<1> {
    using T = uint8_t;
};

template <int V>
union Chunk {
    typename Vec<V>::T v;
    uint8_t b[V];
};

// The label table of byte `off` of band row y.
__device__ __forceinline__ uint8_t label_byte(const SplitArgs &a, int y, int off, uint8_t b) {
    const uint16_t c = __ldg(a.cls + (int64_t)y * a.W + off / 3);
    return c ? __ldg(a.lut + ((int)c << 8) + b) : b;
}

// One byte of the output row, from scratch (boundary chunks, row tails, and the V = 1 path).
__device__ __forceinline__ uint8_t compose_byte(const SplitArgs &a, const uint8_t *lrow, const uint8_t *rrow, int y, int off) {
    uint8_t b = off < a.split ? lrow[off] : rrow[off];
    if (a.seam && off >= a.split && off < a.split + 3) b = 255;
    if (y < a.band_rows) b = label_byte(a, y, off, b);
    return b;
}

template <int V>
__global__ void __launch_bounds__(THREADS, MIN_CTAS) split_compose_kernel(SplitArgs a) {
    using T = typename Vec<V>::T;
    const int c0 = blockIdx.x * CHUNKS_PER_CTA + threadIdx.x;
    for (int f = blockIdx.z; f < a.n; f += gridDim.z) {
        for (int y = blockIdx.y; y < a.H; y += gridDim.y) {
            const uint8_t *lrow = a.left + f * a.lfs + y * a.lrs;
            const uint8_t *rrow = a.right + f * a.rfs + y * a.rrs;
            uint8_t *orow = a.out + f * a.ofs + y * a.ors;
            Chunk<V> ch[UNROLL];
            bool full[UNROLL];
#pragma unroll
            for (int u = 0; u < UNROLL; ++u) {
                const int off = (c0 + u * THREADS) * V;
                full[u] = off + V <= a.row_bytes;
                if (!full[u]) continue;
                if (off + V <= a.split) {
                    ch[u].v = __ldg(reinterpret_cast<const T *>(lrow + off));
                } else if (off >= a.split) {
                    ch[u].v = __ldg(reinterpret_cast<const T *>(rrow + off));
                } else {                                   // the chunk that holds the left/right boundary
                    Chunk<V> l, r;
                    l.v = __ldg(reinterpret_cast<const T *>(lrow + off));
                    r.v = __ldg(reinterpret_cast<const T *>(rrow + off));
#pragma unroll
                    for (int i = 0; i < V; ++i) ch[u].b[i] = off + i < a.split ? l.b[i] : r.b[i];
                }
            }
#pragma unroll
            for (int u = 0; u < UNROLL; ++u) {
                const int off = (c0 + u * THREADS) * V;
                if (!full[u]) {                            // the row's partial last chunk
                    for (int i = off; i < a.row_bytes && i < off + V; ++i) orow[i] = compose_byte(a, lrow, rrow, y, i);
                    continue;
                }
                if (a.seam && off < a.split + 3 && off + V > a.split) {
#pragma unroll
                    for (int i = 0; i < V; ++i)
                        if (off + i >= a.split && off + i < a.split + 3) ch[u].b[i] = 255;
                }
                if (y < a.band_rows) {
#pragma unroll
                    for (int i = 0; i < V; ++i) ch[u].b[i] = label_byte(a, y, off + i, ch[u].b[i]);
                }
                *reinterpret_cast<T *>(orow + off) = ch[u].v;
            }
        }
    }
}

bool aligned(const void *p, int64_t s0, int64_t s1, int v) {
    return ((uintptr_t)p % v) == 0 && s0 % v == 0 && s1 % v == 0;
}

}  // namespace

extern "C" int avb_split_compose_u8(const uint8_t *left, const uint8_t *right, uint8_t *out, int n, int H, int W,
                                    int64_t left_frame_stride, int64_t left_row_stride, int64_t right_frame_stride,
                                    int64_t right_row_stride, int64_t out_frame_stride, int64_t out_row_stride, int seam,
                                    int band_rows, const uint16_t *classes_dev, const uint8_t *luts_dev,
                                    avb_stream_t stream) {
    AVB_REQUIRE(left && right && out, "null frame pointer");
    AVB_REQUIRE(n >= 1 && H >= 1 && W >= 1, "n, H and W must be positive");
    AVB_REQUIRE(3LL * W <= (1LL << 30), "rows longer than 2^30 bytes");
    AVB_REQUIRE(left_row_stride >= 3LL * W && right_row_stride >= 3LL * W && out_row_stride >= 3LL * W,
                "row strides must be at least 3 * W bytes");
    AVB_REQUIRE(left_frame_stride >= 0 && right_frame_stride >= 0, "negative frame stride");
    AVB_REQUIRE(n == 1 || out_frame_stride >= out_row_stride * (H - 1) + 3LL * W, "output frames overlap");
    AVB_REQUIRE(band_rows >= 0 && band_rows <= H, "band_rows must lie in [0, H]");
    AVB_REQUIRE(band_rows == 0 || (classes_dev && luts_dev), "a label band needs its class map and tables");
    SplitArgs a;
    a.left = left;
    a.right = right;
    a.out = out;
    a.lfs = left_frame_stride;
    a.lrs = left_row_stride;
    a.rfs = right_frame_stride;
    a.rrs = right_row_stride;
    a.ofs = out_frame_stride;
    a.ors = out_row_stride;
    a.n = n;
    a.H = H;
    a.W = W;
    a.row_bytes = 3 * W;
    a.split = 3 * (W / 2);
    a.seam = seam != 0;
    a.band_rows = band_rows;
    a.cls = classes_dev;
    a.lut = luts_dev;
    const bool v16 = aligned(left, a.lfs, a.lrs, 16) && aligned(right, a.rfs, a.rrs, 16) && aligned(out, a.ofs, a.ors, 16);
    const bool v4 = aligned(left, a.lfs, a.lrs, 4) && aligned(right, a.rfs, a.rrs, 4) && aligned(out, a.ofs, a.ors, 4);
    const int V = v16 ? 16 : v4 ? 4 : 1;
    const int chunks = (a.row_bytes + V - 1) / V;
    const dim3 grid((chunks + CHUNKS_PER_CTA - 1) / CHUNKS_PER_CTA, H < 65535 ? H : 65535, n < 65535 ? n : 65535);
    cudaStream_t st = (cudaStream_t)stream;
    {
        AVB_TIMED("split_compose", st);
        if (V == 16)
            split_compose_kernel<16><<<grid, THREADS, 0, st>>>(a);
        else if (V == 4)
            split_compose_kernel<4><<<grid, THREADS, 0, st>>>(a);
        else
            split_compose_kernel<1><<<grid, THREADS, 0, st>>>(a);
    }
    AVB_CUDA_OK(cudaGetLastError());
    return AVB_OK;
}

// The bytes of a composed split frame that can differ from its input frame, device -> host: rows [0, band_rows) whole,
// and bytes [3 * (W / 2), 3W) of rows [band_rows, H) (the seam and the right half).  Everything else is the left half of
// the input outside the label band, so fetching into the host frames that were uploaded turns them into their split
// frames.  Pitched copies, two per frame, or two in all when both sides stack their frames as whole rows (one 3D copy
// per piece).  The destination must be page-locked: a pageable one would make the copy synchronous and staged.
namespace {

// Frames lie `frame_stride / row_stride` whole rows apart, so a 3D copy with that slice height reaches every frame.
bool stacked(int64_t frame_stride, int64_t row_stride, int H) {
    return frame_stride % row_stride == 0 && frame_stride / row_stride >= H;
}

cudaError_t memory_type(const void *p, cudaMemoryType *type) {
    cudaPointerAttributes at = {};
    const cudaError_t e = cudaPointerGetAttributes(&at, p);
    *type = at.type;
    return e;
}

}  // namespace

extern "C" int avb_split_fetch_u8(const uint8_t *src, uint8_t *dst_host, int n, int H, int W, int64_t src_frame_stride,
                                  int64_t src_row_stride, int64_t dst_frame_stride, int64_t dst_row_stride, int band_rows,
                                  avb_stream_t stream) {
    AVB_REQUIRE(src && dst_host, "null frame pointer");
    AVB_REQUIRE(n >= 1 && H >= 1 && W >= 1, "n, H and W must be positive");
    AVB_REQUIRE(3LL * W <= (1LL << 30), "rows longer than 2^30 bytes");
    AVB_REQUIRE(src_row_stride >= 3LL * W && dst_row_stride >= 3LL * W, "row strides must be at least 3 * W bytes");
    AVB_REQUIRE(src_frame_stride >= 0, "negative frame stride");
    AVB_REQUIRE(n == 1 || dst_frame_stride >= dst_row_stride * (H - 1) + 3LL * W, "destination frames overlap");
    AVB_REQUIRE(band_rows >= 0 && band_rows <= H, "band_rows must lie in [0, H]");
    const int64_t src_last = (n - 1) * src_frame_stride + (H - 1) * src_row_stride + 3LL * W - 1;
    const int64_t dst_last = (n - 1) * dst_frame_stride + (H - 1) * dst_row_stride + 3LL * W - 1;
    cudaMemoryType type;                      // first and last byte of each side
    for (const uint8_t *p : {src, src + src_last}) {
        AVB_CUDA_OK(memory_type(p, &type));
        AVB_REQUIRE(type == cudaMemoryTypeDevice, "src must be device memory");
    }
    for (const uint8_t *p : {(const uint8_t *)dst_host, (const uint8_t *)dst_host + dst_last}) {
        AVB_CUDA_OK(memory_type(p, &type));
        AVB_REQUIRE(type == cudaMemoryTypeHost, "dst_host must be page-locked host memory (a pageable destination "
                                                "makes the copy synchronous and staged)");
    }
    const int64_t row = 3LL * W, split = 3LL * (W / 2);
    struct Piece {
        int y0, rows;
        int64_t x0, width;
    };
    const Piece pieces[2] = {{0, band_rows, 0, row}, {band_rows, H - band_rows, split, row - split}};
    const bool one_copy = stacked(src_frame_stride, src_row_stride, H) && stacked(dst_frame_stride, dst_row_stride, H);
    cudaStream_t st = (cudaStream_t)stream;
    for (const Piece &p : pieces) {
        if (p.rows == 0) continue;
        if (one_copy) {
            cudaMemcpy3DParms c = {};
            c.srcPtr = make_cudaPitchedPtr((void *)src, src_row_stride, row, src_frame_stride / src_row_stride);
            c.dstPtr = make_cudaPitchedPtr(dst_host, dst_row_stride, row, dst_frame_stride / dst_row_stride);
            c.srcPos = c.dstPos = make_cudaPos(p.x0, p.y0, 0);
            c.extent = make_cudaExtent(p.width, p.rows, n);
            c.kind = cudaMemcpyDeviceToHost;
            AVB_CUDA_OK(cudaMemcpy3DAsync(&c, st));
        } else {
            for (int f = 0; f < n; ++f) {
                const int64_t so = f * src_frame_stride + p.y0 * src_row_stride + p.x0;
                const int64_t doff = f * dst_frame_stride + p.y0 * dst_row_stride + p.x0;
                AVB_CUDA_OK(cudaMemcpy2DAsync(dst_host + doff, dst_row_stride, src + so, src_row_stride, p.width, p.rows,
                                              cudaMemcpyDeviceToHost, st));
            }
        }
    }
    return AVB_OK;
}
