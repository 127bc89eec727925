/* avb200.h -- C ABI of libavb200.so: the B200 (sm_100a) pixel pipeline behind animal-vision's
 * `Animal.visualize()`.
 *
 * Every entry point replaces a piece of the reference's per-frame NumPy/OpenCV/torch code path
 * (cited per function as file:line under the reference tree).  Conventions:
 *   - frames are packed 8-bit, 3 interleaved channels, addressed with explicit BYTE strides
 *     (frame stride, row stride); channel order is never interpreted (the reference is fed RGB by
 *     its renderers and BGR by its server and indexes channels 0/1/2 either way);
 *   - `in`, `out`, `*_dev` pointers are DEVICE pointers owned by the caller (torch); `*_host`
 *     pointers are small host arrays read during the call; nothing is retained after return;
 *   - all work is enqueued on `stream` (a cudaStream_t); no call synchronises the device;
 *   - return value 0 = ok, negative = AVB_E_*; avb_last_error() gives the message of the last
 *     failure on the calling thread.
 * There is no CPU fallback: with no CUDA device every compute entry point returns AVB_E_CUDA.
 */
#ifndef AVB200_H
#define AVB200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AVB_VERSION 170            /* 0.1.7 */

#define AVB_OK 0
#define AVB_E_ARG (-1)             /* bad argument (null pointer, non-positive size, unsupported radius ...) */
#define AVB_E_CUDA (-2)            /* CUDA runtime error (message in avb_last_error) */
#define AVB_E_UNSUPPORTED (-3)

/* How the 8-bit input is normalised before the sRGB decode. */
#define AVB_NORM_DIV255 0          /* uv_helpers.py:15-19 to_float01: uint8 is always divided by 255 */
#define AVB_NORM_AUTO 1            /* animals/animal_utils.py:41-50 get_normalized_image: divide by 255
                                      only if the frame maximum exceeds 1 (decided per frame, on device) */

typedef void *avb_stream_t;        /* cudaStream_t */

#if defined(__GNUC__)
#define AVB_API __attribute__((visibility("default")))
#else
#define AVB_API
#endif

AVB_API int avb_version(void);
AVB_API const char *avb_last_error(void);
/* First 16 hex digits of the SHA-256 of the include/avb200.h this library was compiled against: a binding
 * compares it with its own copy of the header before typing any symbol, so that a stale binary whose
 * argument lists differ is refused instead of being called with the wrong stack layout. */
AVB_API const char *avb_header_sha(void);

/* Per-kernel timing for benchmarks.  After avb_profile_begin(), every kernel the library launches
 * from the calling thread is bracketed by CUDA events on its stream; avb_profile_end() waits for
 * them and returns up to `capacity` (name, milliseconds) records in launch order (names are
 * NUL-terminated strings `name_stride` bytes apart).  Returns the number of records. */
AVB_API int avb_profile_begin(void);
AVB_API int avb_profile_end(char *names, int name_stride, float *ms, int capacity);

/* Number of uint32 entries avb_build_encode_table writes at most. */
#define AVB_ENC_TABLE_MAX 2048

/* Host helper.  Turns the 255 quantisation thresholds of the reference's encode tail
 * (clip -> linear_to_srgb -> clip -> x*255+0.5 -> astype(uint8); animals/dog.py:54-59 with
 * animals/animal_utils.py:13-19) into the bucketed lookup table the kernels use.
 *   thr_host[i-1] = smallest float32 x in [0,1] whose encoded byte is >= i, i = 1..255
 * (built by the host with the reference's own NumPy expression, so the device quantiser IS the
 * reference's step function).  Writes table_host[0..n) (n <= AVB_ENC_TABLE_MAX) and returns n, or
 * a negative error.  The caller uploads the table and passes the device pointer as `enc_dev`. */
AVB_API int avb_build_encode_table(const float *thr_host, uint32_t *table_host, int capacity);

/* K1 -- fused per-pixel colorimetric kernel (HBM bound, 6 B/px).
 * Replaces animals/animal_utils.py:41-50 (normalise), :5-11 (sRGB decode), the `pixels @ T.T`
 * 3x3 of animals/dog.py:44-48 with T from animal_utils.py:88-119, the optional per-row S-cone gain
 * of animal_utils.py:206-259 (rat.py:34), and the encode tail dog.py:54-59.
 *   dec_dev      256 float32 decode LUT for frames that are divided by 255
 *   dec_raw_dev  256 float32 decode LUT for frames whose max is <= 1 (AVB_NORM_AUTO only; may be NULL
 *                with AVB_NORM_DIV255)
 *   enc_dev      table from avb_build_encode_table
 *   m_host       9 floats, row-major T; out[c] = sum_k T[c][k] * lin[k]
 *   row_gain_dev NULL, or H floats: channel 2 is multiplied by row_gain[y] and clipped to [0,1]
 *   flags_dev    n uint32 scratch words (AVB_NORM_AUTO only) */
AVB_API int avb_colorimetric_u8(const uint8_t *in, uint8_t *out, int n, int H, int W,
                        int64_t in_frame_stride, int64_t in_row_stride,
                        int64_t out_frame_stride, int64_t out_row_stride,
                        const float *dec_dev, const float *dec_raw_dev, const uint32_t *enc_dev,
                        const float *m_host, const float *row_gain_dev,
                        int norm_mode, uint32_t *flags_dev, avb_stream_t stream);

/* K2 -- dichromat recipe with an isotropic acuity blur, one fused kernel:
 * decode -> 3x3 -> separable Gaussian (BORDER_REFLECT_101) -> clip -> encode.
 * Replaces animals/dog.py:35-59 (and the 8 sibling species that call apply_acuity_blur,
 * animals/animal_utils.py:121-145 = cv2.GaussianBlur(img,(0,0),sigma)).
 *   taps_host    ksize float32 taps (cv2.getGaussianKernel(ksize, sigma, CV_32F)), ksize odd, <= 33 */
AVB_API int avb_dichromat_blur_u8(const uint8_t *in, uint8_t *out, int n, int H, int W,
                          int64_t in_frame_stride, int64_t in_row_stride,
                          int64_t out_frame_stride, int64_t out_row_stride,
                          const float *dec_dev, const float *dec_raw_dev, const uint32_t *enc_dev,
                          const float *m_host, const float *taps_host, int ksize,
                          int norm_mode, uint32_t *flags_dev, avb_stream_t stream);

/* K2s -- dichromat recipe with the per-row "streak" blur of the grazing mammals, one fused kernel:
 * decode -> per-row 3x3 -> per-row horizontal correlation -> [chroma compression] -> clip -> encode.
 * Replaces animals/cow.py:25-45 (and deer, goat, horse, kangaroo, sheep, panda, rabbit, pig), i.e.
 * apply_anisotropic_acuity_blur_with_streak (animals/animal_utils.py:147-172) as it actually behaves
 * (x blur + 3-wide colour-channel leak with sigmaX(y), x blur with sigmaY(y), never any vertical
 * blur) and apply_chroma_compression (animal_utils.py:174-181).
 *   row_tab_dev     H x 56 float32 (host-built: animal_vision_b200/tables.py streak_row_table):
 *                   [0:33] combined x taps centred at 16, [33:42] row-major 3x3 (channel mix @ species
 *                   matrix), [42] combined radius (<= 16), [43:55] the rank-2 factors (3x2 P_y, 2x3 Q), [55] 1 when valid; 56 floats per row
 *   chroma_strength 0 = no chroma compression (panda/rabbit: 0.06) */
AVB_API int avb_streak_blur_u8(const uint8_t *in, uint8_t *out, int n, int H, int W,
                               int64_t in_frame_stride, int64_t in_row_stride,
                               int64_t out_frame_stride, int64_t out_row_stride,
                               const float *dec_dev, const float *dec_raw_dev, const uint32_t *enc_dev,
                               const float *row_tab_dev, float chroma_strength,
                               int norm_mode, uint32_t *flags_dev, avb_stream_t stream);

/* Cat -- both outputs of Cat.visualize (animals/cat.py:73-114, the runnable side of the merge
 * conflict) for a batch of frames:
 *   out_human  centre zoom (animals/cat_widevision_utils.py:11-29: crop + cv2.resize INTER_LINEAR on
 *              uint8, restated in OpenCV's 11-bit fixed point, bit-exact); may be NULL with zoom_dev NULL
 *   out_cat    binocular wide-FOV warp (cat_widevision_utils.py:46-99; cv2.remap INTER_LINEAR with its
 *              1/32-px coordinate quantisation, BORDER_CONSTANT 0, cos^2 blend) fused, as the producer
 *              stage, into the K2 blur kernel: decode (pow) -> collapsed 3x3 (cat.py:95-101) ->
 *              Gaussian sigma=1.0 (9 taps) -> encode.
 *   dec_dev / dec_raw_dev  decode LUTs as in avb_colorimetric_u8; only read when warp_dev is NULL
 *   warp_dev   NULL = class switch ENABLE_FOV_WARP False (cat.py:21): no warp, LUT producer; else
 *              6*W float32: xL, xR, wL, wR (per-column source x of the two eye views, blend weights),
 *              ws = wL + wR + 1e-8 (the blend denominator, float32) and 1/ws (correctly rounded)
 *   zoom_dev   4*W + 4*H int32, 16-byte aligned: W records {xi0, xi1, xw0, xw1} then H records
 *              {yi0, yi1, yw0, yw1} (source indices incl. crop origin, 11-bit weights)
 *   enc_dev    encode table built from the float64 tail's thresholds (cat.py runs float64 from
 *              LMS_to_RGB on; the device tail is float32, SURVEY.md 8a-9)
 *   flags_dev  n uint32 scratch (AVB_NORM_AUTO): filled by a pre-pass over each frame */
AVB_API int avb_cat_u8(const uint8_t *in, uint8_t *out_human, uint8_t *out_cat, int n, int H, int W,
                       int64_t in_frame_stride, int64_t in_row_stride,
                       int64_t human_frame_stride, int64_t human_row_stride,
                       int64_t cat_frame_stride, int64_t cat_row_stride,
                       const float *dec_dev, const float *dec_raw_dev,
                       const uint32_t *enc_dev, const float *m_host, const float *taps_host, int ksize,
                       const float *warp_dev, const int32_t *zoom_dev,
                       int norm_mode, uint32_t *flags_dev, avb_stream_t stream);

/* K3 -- the UV path, HoneyBee.visualize (animals/honeybee.py:99-175):
 * RGB -> analytic 31-band spectrum (ml/classic_rgb_to_hsi/classic_rgb_to_hsi.py:47-82) -> x illuminant
 * (uv_helpers.py:187-192) -> three receptor catches (honeybee.py:133-135) -> von Kries adaptation
 * (uv_helpers.py:195-206) -> acuity blur (uv_helpers.py:67-73) -> (U,B,G) visualisation map with its
 * global percentiles (uv_mappers.py:29-144) -> clip -> OETF -> uint8 (honeybee.py:166-173).
 * The H x W x B cube is never written: catches are (re)computed per pixel in registers; the
 * percentiles are the exact order statistics numpy.percentile(method="linear") interpolates.
 *   dec_dev        256 float32 decode LUT (uint8 -> /255 -> torch sRGB decode)
 *   m3_host        9 floats: catches = M3 @ lin  (spectral chain collapsed to 3x3); used when n_bands == 0
 *   bands_dev      n_bands x 8 float32 rows {g0,g1,g2, E, s0,s1,s2, 0}: lobe of input channel c,
 *                  illuminant, receptor sensitivities; n_bands > 0 selects the per-pixel band loop
 *   denom_eps      lobe normaliser + 1e-8 (float32)
 *   adapt_mode     0 none, 1 white patch (global max), 2 gray world (global mean)
 *   blur_taps_host ksize taps (ksize 0, 3 or 5)
 *   map_mode       AVB_MAP_*: uv_mappers.py map_opponent :53-64 (P95 radius, P95 L), map_falsecolor
 *                  :29-43 (P95 x3), map_linear_matrix :45-50, map_uv_purple_yellow_soft :90-132 (P98),
 *                  map_falsecolor_uv_mixed :135-144
 *   map_params_host 15 floats (may be NULL for opponent / falsecolor): [0:9] row-major matrix of
 *                  AVB_MAP_MATRIX, [9:12] / [12:15] linear-light purple / warm anchors of the
 *                  purple-yellow map (uv_mappers.py:107-116, evaluated by the host in NumPy)
 *   mix_alpha      blend weight of AVB_MAP_MIXED (honeybee.py:161 passes 0.45)
 *   workspace_dev  avb_uv_workspace_bytes(n, H, W, map_mode) bytes of scratch, 16-byte aligned
 *   dbg_catches_dev NULL, or n*H*W*3 float32: raw receptor catches (test hook for the 1e-5 check) */
#define AVB_MAP_OPPONENT 0
#define AVB_MAP_FALSECOLOR 1
#define AVB_MAP_MATRIX 2
#define AVB_MAP_PURPLE_YELLOW 3
#define AVB_MAP_MIXED 4
AVB_API int64_t avb_uv_workspace_bytes(int n, int H, int W, int map_mode);
AVB_API int avb_uv_map_u8(const uint8_t *in, uint8_t *out, int n, int H, int W,
                          int64_t in_frame_stride, int64_t in_row_stride,
                          int64_t out_frame_stride, int64_t out_row_stride,
                          const float *dec_dev, const uint32_t *enc_dev,
                          const float *m3_host, const float *bands_dev, int n_bands, float denom_eps,
                          int adapt_mode, const float *blur_taps_host, int blur_ksize,
                          int map_mode, const float *map_params_host, float mix_alpha,
                          void *workspace_dev, float *dbg_catches_dev, avb_stream_t stream);

/* K4 -- MST++ RGB -> 31-band hyperspectral inference (reference
 * ml/MST_plus_plus/predict_code/architecture/MST_Plus_Plus.py:270-293 MST_Plus_Plus.forward, wrapper
 * semantics of ml/MST_plus_plus/predict_code/predict_torch.py:249-310).
 *   avb_mstpp_create   params_host: the 1 619 625 float32 values of MST_Plus_Plus().state_dict() (227
 *                      tensors, registration order, native layouts); padded / permuted / cast to bf16
 *                      and uploaded once.  Replaces architecture/__init__.py:36-40 (weight loading).
 *   avb_mstpp_forward  in: device [n,H,W,3] float32 in [0,1] (in_is_u8 = 0) or uint8 (in_is_u8 = 1,
 *                      divided by 255: predict_torch.py:12-19); out: device float32 [n,H,W,31].
 *                      pad_multiple / centred choose the reflect padding: (8, 0) = the model's own
 *                      bottom/right pad (MST_Plus_Plus.py:284-288), (16, 1) = the wrapper's centred pad
 *                      (predict_torch.py:171-188).
 *   workspace_dev      avb_mstpp_workspace_bytes(n, H, W, pad_multiple, centred) bytes */
AVB_API int avb_mstpp_create(const float *params_host, int64_t count, void **handle);
AVB_API int avb_mstpp_destroy(void *handle);
AVB_API int64_t avb_mstpp_workspace_bytes(int n, int H, int W, int pad_multiple, int centred);
AVB_API int avb_mstpp_forward(void *handle, const void *in, int in_is_u8, float *out, int n, int H, int W,
                              int pad_multiple, int centred, void *workspace_dev, avb_stream_t stream);
/* The same forward with the band projection of `integrate_band` (uv_helpers.py:142-146) FUSED on the network output
 * (BASELINE config 4: "mantis shrimp multi-receptor projection via MST++"): bands_out [n,H,W,n_bands] float32 =
 * cube . band_weights^T, band_weights_dev [n_bands][31] (e.g. the ten raised-cosine bands of mantis_shrimp.py:49-60),
 * evaluated in the epilogue of conv_out from the accumulator registers.  out may be NULL: the 31-band cube is then never
 * written (30 MB per 482x512 patch).  bands_out = NULL, n_bands = 0 is avb_mstpp_forward. */
AVB_API int avb_mstpp_forward_bands(void *handle, const void *in, int in_is_u8, float *out, float *bands_out,
                                    const float *band_weights_dev, int n_bands, int n, int H, int W,
                                    int pad_multiple, int centred, void *workspace_dev, avb_stream_t stream);

/* Spectral band projection out[px][r] = sum_b cube[px][b] * weights[r][b] -- np.tensordot over the band
 * axis as in uv_helpers.py:142-146 integrate_band and animals/mantis_shrimp.py:49-60 (ten bands);
 * weights come from the host (uv_helpers.py:125-139 bandpass_weights).  All pointers device float32. */
AVB_API int avb_band_project_f32(const float *cube_dev, const float *weights_dev, float *out_dev,
                                 int64_t npx, int n_bands, int n_receptors, avb_stream_t stream);

/* uv_helpers.py:47-53 safe_norm on n_maps interleaved float32 maps (element px of map k at
 * in[px*stride + k]): (x - min) / (max - min) over the whole map, zeros when max - min < 1e-9.
 * scratch_dev: 2*n_maps uint32.  In place (out_dev == in_dev) is allowed. */
AVB_API int avb_safe_norm_f32(const float *in_dev, float *out_dev, int64_t npx, int stride, int n_maps,
                              void *scratch_dev, avb_stream_t stream);

/* Float-frame path of the 19 dichromat mammals: "float in => float [0,1] out, no quantisation"
 * (animals/dog.py:56-59).  get_normalized_image's branch (animals/animal_utils.py:41-50: divide by
 * 255 only if the frame maximum exceeds 1) is decided per frame on the device; decode / encode are
 * the IEC 61966-2-1 functions of animal_utils.py:5-19 in float32.  All frame pointers: packed device
 * float32 [n,H,W,3]; `tmp_dev` is scratch of the same size; `out_dev` must not alias `in_dev`.
 *   kind          AVB_F32_POINT   no spatial filter (Rat: row_gain_dev = S-cone gain per row, or NULL)
 *                 AVB_F32_GAUSS   cv2.GaussianBlur taps (host, odd ksize <= 33), REFLECT_101
 *                                 (animal_utils.py:121-145)
 *                 AVB_F32_STREAK  per-row filter, row_tab_dev as for avb_streak_blur_u8
 *                                 (animal_utils.py:147-172)
 *   chroma        apply_chroma_compression strength after the filter (animal_utils.py:174-181), 0 = off
 *   quantize      1: finish with trunc(x*255 + 0.5) for callers whose frames had an integer dtype
 *                 other than uint8 (dog.py:56-57); the values stay float32
 *   maxbits_dev   n uint32 of scratch */
#define AVB_F32_POINT 0
#define AVB_F32_GAUSS 1
#define AVB_F32_STREAK 2
AVB_API int avb_dichromat_f32(const float *in_dev, float *out_dev, float *tmp_dev, int n, int H, int W,
                              const float *m_host, int kind, const float *taps_host, int ksize,
                              const float *row_tab_dev, const float *row_gain_dev, float chroma, int quantize,
                              uint32_t *maxbits_dev, avb_stream_t stream);

/* ---- K6: generic float32 image operators (csrc/k6_imgops.cu) -------------------------------------
 * The generality route behind the fused uint8 kernels: float / wide-integer frames, HoneyBee's
 * hsi_downsample and large blur sigmas, and the UV species composed from uv_helpers.py steps.
 * Images: device float32, packed [n, H, W, C]. */
#define AVB_IMG_NORM_UV 0          /* uv_helpers.py:15-23 to_float01: uint8 / 255; other dtypes clip(x/255) only if max > 1.001 */
#define AVB_IMG_NORM_MAMMAL 1      /* animals/animal_utils.py:41-50 get_normalized_image: / 255 if max > 1, then clip to [0,1] */
/* in_dev: n frames of per_frame values, uint8 (in_is_u8 = 1) or float32; scratch_dev: n uint32. */
AVB_API int avb_img_to_float01(const void *in_dev, int in_is_u8, float *out_dev, int n, int64_t per_frame, int mode,
                               uint32_t *scratch_dev, avb_stream_t stream);

/* One axis of cv2.resize (uv_helpers.py:57-64 resize_preserve_range, :84-99 panorama_warp, :155-183
 * classic_rgb_to_hsi_scaled; animals/cat_widevision_utils.py:11-29 center_zoom on float frames):
 *   axis 0: out[f][y][x][c] = sum_t w[x][t] * in[f][y][idx[x][t]][c]      (Hout rows of the input are read)
 *   axis 1: out[f][y][x][c] = sum_t w[y][t] * in[f][idx[y][t]][x][c]
 * idx_dev / w_dev: [len(axis)][taps] tables built by the host with OpenCV's own coordinate arithmetic
 * (animal_vision_b200/tables.py resize_taps: INTER_LINEAR, INTER_CUBIC, INTER_AREA); borders are already
 * resolved in idx.  in_frame_stride / in_row_stride are in ELEMENTS (a crop is a pointer offset + strides);
 * the output is contiguous [n, Hout, Wout, C].  OpenCV runs the horizontal pass first. */
AVB_API int avb_img_resample(const float *in_dev, float *out_dev, int n, int Hout, int Wout, int C, int axis,
                             int64_t in_frame_stride, int64_t in_row_stride, const int32_t *idx_dev, const float *w_dev,
                             int taps, avb_stream_t stream);

/* Separable correlation with BORDER_REFLECT_101, rows first: cv2.GaussianBlur(img, (k,k), sigma) as
 * uv_helpers.py:67-73 gaussian_blur calls it (k = 2*ceil(3*sigma)+1; any odd tap count).  taps on the device. */
AVB_API int avb_img_blur(const float *in_dev, float *out_dev, float *tmp_dev, int n, int H, int W, int C,
                         const float *taps_x_dev, int kx, const float *taps_y_dev, int ky, avb_stream_t stream);

/* Per frame and channel {min, max, mean, 0} -> out_dev[n][C][4] (uv_helpers.py:47-53 safe_norm, :195-206 von
 * Kries).  scratch_dev: 16 * n * C bytes. */
#define AVB_STAT_MIN 0
#define AVB_STAT_MAX 1
#define AVB_STAT_MEAN 2
AVB_API int avb_img_stats(const float *in_dev, int n, int64_t npx, int C, float *out_dev, void *scratch_dev, avb_stream_t stream);
/* out = in / max(stats[f][c][which], eps): von_kries_white_patch (AVB_STAT_MAX) / _gray_world (AVB_STAT_MEAN). */
AVB_API int avb_img_divide_channels(const float *in_dev, float *out_dev, int n, int64_t npx, int C, const float *stats_dev,
                                    int which, float eps, avb_stream_t stream);

/* numpy.percentile(x, q) (method "linear", float32 result) of nreq strided planes: request r covers the npx
 * values in_dev[offsets_host[r] + i*stride]; exact (three-level radix select over the float bit patterns, then
 * numpy's interpolation between the two neighbouring order statistics).  Used by uv_mappers.py:29-43,
 * animals/rat_uv.py:171-174 and siblings.  scratch_dev: avb_img_percentile_scratch_bytes(min(nreq,16)). */
AVB_API int64_t avb_img_percentile_scratch_bytes(int nreq);
AVB_API int avb_img_percentile(const float *in_dev, int64_t npx, int64_t stride, const int64_t *offsets_host,
                               const double *q_host, int nreq, float *out_dev, void *scratch_dev, avb_stream_t stream);

/* animals/cat_widevision_utils.py:46-99 animal_fov_binocular_warp on float32 [0,1] frames [n,H,W,3] (the float-frame
 * route of Cat.visualize, animals/cat.py:83-93): both eye views by cv2.remap's 1/32-px bilinear, cos^2 blend, clip.
 * warp_dev: the 6*W table of avb_cat_u8.  out_dev must not alias in01_dev. */
AVB_API int avb_cat_warp_f32(const float *in01_dev, float *out_dev, int n, int H, int W, const float *warp_dev, avb_stream_t stream);

/* Float32 plane route of the UV path (animals/honeybee.py:99-175 for float / wide-integer frames,
 * hsi_downsample = True and blur sigmas beyond the fused walker):
 *   avb_uv_catches_f32  img01 [npx][3] -> sRGB decode (classic_rgb_to_hsi.py:16-22) -> analytic spectrum ->
 *                       illuminant -> raw receptor catches [npx][3] (honeybee.py:126-135); tables as avb_uv_map_u8
 *   avb_uv_map_f32      adapted + blurred (U,B,G) planes [n][H][W][3] -> mapper with its global percentiles
 *                       (uv_mappers.py) -> clip -> OETF -> uint8 frames (strided) or float32 [n][H][W][3]
 *                       (quantize = 1: x*255+0.5 truncated, for integer dtypes other than uint8)
 *   workspace_dev       avb_uv_workspace_bytes(n, H, W, map_mode) bytes */
AVB_API int avb_uv_catches_f32(const float *img01_dev, float *catches_dev, int64_t npx, const float *m3_host,
                               const float *bands_dev, int n_bands, float denom_eps, avb_stream_t stream);
AVB_API int avb_uv_map_f32(const float *ubg_dev, void *out, int out_is_f32, int quantize, int n, int H, int W,
                           int64_t out_frame_stride, int64_t out_row_stride, const uint32_t *enc_dev,
                           int map_mode, const float *map_params_host, float mix_alpha,
                           void *workspace_dev, avb_stream_t stream);

/* ---- K7: fused per-pixel programs + cv2.remap (csrc/k7_pointwise.cu) --------------------------------
 * The element-wise arithmetic of the UV species (animals/reindeer.py:70-135, goldfish.py, damselfish.py,
 * rat_uv.py:131-214, anableps.py:124-255, anchovy.py:130-253, guppy.py:132-235, morpho.py, heliconius.py,
 * pieris.py, kestrel.py:113-234, jumping_spider.py:135-236, dragonfly.py:146-251, hummingbird.py:128-227,
 * mantis_shrimp.py:143-279) runs as register programs: one launch per maximal run of NumPy element-wise steps.
 * Every instruction is one IEEE float32 operation (r = register file, 'a' / 'b' register numbers):
 *   LOAD   r[dst] = src[a] channel b       CONST r[dst] = imm (float bits)     STORE  dst[b] channel imm = r[a]
 *   SELECT r[dst] = r[a] != 0 ? r[b] : r[imm & 255]
 *   QUANT  trunc(clip(x*255 + 0.5, 0, 255))          (uv_helpers.py:26-30 from_float01, integer dtypes)
 *   SRGB_DEC / SRGB_ENC                              (uv_helpers.py:33-44)
 * Sources: float32 planes [n][H*W][pix_stride] (frame_stride = 0 broadcasts one frame), per-row tables
 * [H][pix_stride], per-column tables [W][pix_stride], per-frame scalars [n][frame_stride] (reduction results stay on
 * the device).  Destinations: float32 or uint8, element index frame*frame_stride + y*row_stride + x*pix_stride + ch. */
enum {
    AVB_VM_NOP = 0, AVB_VM_LOAD, AVB_VM_CONST, AVB_VM_MOV, AVB_VM_ADD, AVB_VM_SUB, AVB_VM_MUL, AVB_VM_DIV, AVB_VM_MIN,
    AVB_VM_MAX, AVB_VM_POW, AVB_VM_ATAN2, AVB_VM_GT, AVB_VM_GE, AVB_VM_LT, AVB_VM_LE, AVB_VM_NEG, AVB_VM_ABS,
    AVB_VM_SQRT, AVB_VM_EXP, AVB_VM_SIN, AVB_VM_COS, AVB_VM_FLOOR, AVB_VM_SRGB_DEC, AVB_VM_SRGB_ENC, AVB_VM_QUANT,
    AVB_VM_SELECT, AVB_VM_STORE,
    /* immediate forms: the second operand is the float in `imm` (R*: reversed, imm op r[a]) -- a constant never costs
     * an instruction or a register of its own */
    AVB_VM_ADDI, AVB_VM_SUBI, AVB_VM_RSUBI, AVB_VM_MULI, AVB_VM_DIVI, AVB_VM_RDIVI, AVB_VM_MINI, AVB_VM_MAXI, AVB_VM_POWI,
    AVB_VM_GTI, AVB_VM_GEI, AVB_VM_LTI, AVB_VM_LEI,
    AVB_VM_N_OPS
};
#define AVB_VM_SRC_PLANE 0
#define AVB_VM_SRC_ROW 1
#define AVB_VM_SRC_COL 2
#define AVB_VM_SRC_FRAME 3
#define AVB_VM_DST_F32 0
#define AVB_VM_DST_U8 1
#define AVB_VM_MAX_SRC 24
#define AVB_VM_MAX_DST 4
#define AVB_VM_MAX_REGS 48
#define AVB_VM_MAX_INS 2048
typedef struct { uint8_t op, dst, a, b; uint32_t imm; } avb_vm_ins;
typedef struct { const void *ptr; int64_t frame_stride; int32_t pix_stride; int32_t kind; } avb_vm_src;
typedef struct { void *ptr; int64_t frame_stride; int64_t row_stride; int32_t pix_stride; int32_t kind; } avb_vm_dst;
AVB_API int avb_vm_run(const avb_vm_ins *prog_dev, int n_ins, int n_regs, int n, int H, int W,
                       const avb_vm_src *src_host, int n_src, const avb_vm_dst *dst_host, int n_dst, avb_stream_t stream);
/* cv2.remap(src, map_x, map_y, INTER_LINEAR, BORDER_REFLECT_101) on float32 [n,H,W,C] with float32 maps [H,W]
 * (animals/anableps.py:224-237): map coordinates quantised to 1/32 px exactly as OpenCV does. */
AVB_API int avb_img_remap(const float *in_dev, float *out_dev, int n, int H, int W, int C, const float *mapx_dev,
                          const float *mapy_dev, avb_stream_t stream);

/* ---- K8: baseline JPEG encode (csrc/k8_jpeg.cu) ---------------------------------------------------------
 * The bytes of cv2.imencode(".jpg", frame, [IMWRITE_JPEG_QUALITY, q]) with OpenCV's defaults (libjpeg-turbo:
 * baseline, 4:2:0, standard Huffman tables, no restart interval) for n packed 8-bit 3-channel frames in the channel
 * order cv2 expects (BGR); replaces the host encode of the reference's processimage (utils.py:133-199).
 *   header_host     the bytes before the entropy-coded data (SOI .. SOS; animal_vision_b200/tables.py jpeg_header),
 *                   header_len <= AVB_JPEG_HEADER_MAX; copied in front of every frame's data
 *   qtables_host    2 x 64 quantiser values in zigzag order (luma, chroma; the DQT payloads of the header), 1..255
 *   out             n slots of out_slot_stride >= avb_jpeg_bound_bytes(H, W) bytes: frame f's file is written from
 *                   out + f * out_slot_stride, its length (header + data + EOI) to out_lengths_dev[f] (device int64)
 *   workspace_dev   avb_jpeg_workspace_bytes(n, H, W) bytes, 16-byte aligned
 * H and W lie in [1, 65535] (the SOF0 fields). */
#define AVB_JPEG_HEADER_MAX 1024
AVB_API int64_t avb_jpeg_bound_bytes(int H, int W);
AVB_API int64_t avb_jpeg_workspace_bytes(int n, int H, int W);
AVB_API int avb_jpeg_encode_u8(const uint8_t *in, int n, int H, int W, int64_t in_frame_stride, int64_t in_row_stride,
                               const uint8_t *header_host, int header_len, const uint8_t *qtables_host, uint8_t *out,
                               int64_t out_slot_stride, int64_t *out_lengths_dev, void *workspace_dev, avb_stream_t stream);
/* The same for frames in RGB order: the bytes of cv2.imencode(".jpg", frame[..., ::-1], [IMWRITE_JPEG_QUALITY, q]).
 * Arguments as avb_jpeg_encode_u8. */
AVB_API int avb_jpeg_encode_rgb_u8(const uint8_t *in, int n, int H, int W, int64_t in_frame_stride,
                                   int64_t in_row_stride, const uint8_t *header_host, int header_len,
                                   const uint8_t *qtables_host, uint8_t *out, int64_t out_slot_stride,
                                   int64_t *out_lengths_dev, void *workspace_dev, avb_stream_t stream);
/* Optimized Huffman tables: the bytes of cv2.imencode(".jpg", frame, [IMWRITE_JPEG_QUALITY, q, IMWRITE_JPEG_OPTIMIZE, 1])
 * (libjpeg's jpeg_gen_optimal_table on each frame's own symbol counts; the same pixels, usually a smaller file).  Each
 * frame's four DHT segments are built and written on the device; no host synchronisation.
 *   prefix_host     the bytes before the DHT segments (SOI .. SOF0; animal_vision_b200/tables.py jpeg_header_prefix)
 *   sos_host        the SOS segment (tables.py JPEG_SOS); prefix_len, sos_len >= 2 and
 *                   prefix_len + sos_len + 432 <= AVB_JPEG_HEADER_MAX (432: the four DHT segments at most)
 *   workspace_dev   avb_jpeg_opt_workspace_bytes(n, H, W) bytes, 16-byte aligned
 * Other arguments, the slots and the lengths as avb_jpeg_encode_u8; avb_jpeg_bound_bytes bounds a slot. */
AVB_API int64_t avb_jpeg_opt_workspace_bytes(int n, int H, int W);
AVB_API int avb_jpeg_opt_encode_u8(const uint8_t *in, int n, int H, int W, int64_t in_frame_stride,
                                   int64_t in_row_stride, const uint8_t *prefix_host, int prefix_len,
                                   const uint8_t *sos_host, int sos_len, const uint8_t *qtables_host, uint8_t *out,
                                   int64_t out_slot_stride, int64_t *out_lengths_dev, void *workspace_dev,
                                   avb_stream_t stream);
/* The same for frames in RGB order (cv2.imencode of frame[..., ::-1] with IMWRITE_JPEG_OPTIMIZE). */
AVB_API int avb_jpeg_opt_encode_rgb_u8(const uint8_t *in, int n, int H, int W, int64_t in_frame_stride,
                                       int64_t in_row_stride, const uint8_t *prefix_host, int prefix_len,
                                       const uint8_t *sos_host, int sos_len, const uint8_t *qtables_host, uint8_t *out,
                                       int64_t out_slot_stride, int64_t *out_lengths_dev, void *workspace_dev,
                                       avb_stream_t stream);

/* ---- K11: Motion-JPEG AVI records (csrc/k11_mjpeg.cu) ----------------------------------------------------------
 * Packs n encoded files, file f at slots + f * slot_stride and lengths_dev[f] bytes long (device int64, e.g. the slots
 * and lengths of avb_jpeg_encode_u8), contiguously into `out` as AVI '00dc' chunks: the fourcc, a little-endian u32
 * size, the file, then zero bytes up to a multiple of 4 (the size counts them, as OpenCV's AVI writer does).  Record f
 * starts at out + out_offsets_dev[f] (device int64); out_offsets_dev[n] is the bytes written.  `out` holds at least
 * n * (8 + ((slot_stride + 3) & ~3)) bytes; a length outside [0, slot_stride] is clamped to it.  slots is 4-byte, out
 * 16-byte aligned; n lies in [1, 65535]. */
AVB_API int avb_mjpeg_pack_u8(const uint8_t *slots, int64_t slot_stride, const int64_t *lengths_dev, int n, uint8_t *out,
                              int64_t *out_offsets_dev, avb_stream_t stream);

/* ---- K10: PNG encode (csrc/k10_png.cu) -----------------------------------------------------------------
 * The bytes of cv2.imencode(".png", frame) with OpenCV's defaults (libpng 1.6 + zlib: filter Sub, deflate level 1,
 * strategy Z_RLE, memLevel 8, IDAT payloads of 8192 bytes) for n packed BGR uint8 frames of H x W, any byte strides.
 * Stream-ordered on `stream`, never synchronises; everything after the frames (filter, parse, trees, emission,
 * Adler-32, framing, CRC-32) runs on the device.
 *   header_host     the signature, the IHDR chunk and the zlib CMF / FLG bytes (animal_vision_b200/tables.py
 *                   png_header), exactly AVB_PNG_HEADER_LEN bytes
 *   out             n slots of out_slot_stride >= avb_png_bound_bytes(H, W) bytes: frame f's file is written from
 *                   out + f * out_slot_stride, its length to out_lengths_dev[f] (device int64)
 *   workspace_dev   avb_png_workspace_bytes(n, H, W) bytes, 16-byte aligned
 * H and W lie in [1, 65535]. */
#define AVB_PNG_HEADER_LEN 35
AVB_API int64_t avb_png_bound_bytes(int H, int W);
AVB_API int64_t avb_png_workspace_bytes(int n, int H, int W);
AVB_API int avb_png_encode_u8(const uint8_t *in, int n, int H, int W, int64_t in_frame_stride, int64_t in_row_stride,
                              const uint8_t *header_host, int header_len, uint8_t *out, int64_t out_slot_stride,
                              int64_t *out_lengths_dev, void *workspace_dev, avb_stream_t stream);

/* ---- K9: labelled split-compare compose (csrc/k9_split.cu) ---------------------------------------------------
 * make_split_frame (reference renderers/video.py:198-245) for n packed 8-bit 3-channel frames of H x W: columns
 * [0, W/2) of out from left, [W/2, W) from right, column W/2 set to 255 when seam != 0; then, in rows [0, band_rows),
 * every byte b of pixel (y, x) becomes luts_dev[classes_dev[y * W + x] * 256 + b] (class 0 is the identity table).
 * The tables are the corner labels of draw_split_labels (animal_vision_b200/tables.py split_label_stencil); every class
 * index must be below the number of tables.  Strides are in bytes; input frame strides may be 0 (one frame for all),
 * output frames must not overlap, and out must not overlap either input.  band_rows = 0 takes no tables. */
AVB_API int avb_split_compose_u8(const uint8_t *left, const uint8_t *right, uint8_t *out, int n, int H, int W,
                                 int64_t left_frame_stride, int64_t left_row_stride, int64_t right_frame_stride,
                                 int64_t right_row_stride, int64_t out_frame_stride, int64_t out_row_stride, int seam,
                                 int band_rows, const uint16_t *classes_dev, const uint8_t *luts_dev, avb_stream_t stream);

/* The device -> host copy of the bytes of n composed split frames (`src`, device, e.g. avb_split_compose_u8's out) that
 * can differ from their input frames: rows [0, band_rows) at full width, and bytes [3 * (W / 2), 3W) of rows
 * [band_rows, H).  Fetched into the page-locked host frames that were uploaded as the compose's left input, it turns
 * them into their split frames; n * (band_rows * 3W + (H - band_rows) * (3W - 3 * (W / 2))) bytes cross.  Pitched
 * copies (cudaMemcpy3DAsync / cudaMemcpy2DAsync): two in all when both sides keep frame_stride a multiple of row_stride
 * and at least H rows, else two per frame.  Strides are in bytes; destination frames must not overlap.  dst_host must be
 * page-locked host memory and src device memory (cudaPointerGetAttributes of the first and last byte), else AVB_E_ARG. */
AVB_API int avb_split_fetch_u8(const uint8_t *src, uint8_t *dst_host, int n, int H, int W, int64_t src_frame_stride,
                               int64_t src_row_stride, int64_t dst_frame_stride, int64_t dst_row_stride, int band_rows,
                               avb_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* AVB200_H */
