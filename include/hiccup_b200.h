/* hiccup_b200.h -- C ABI of the B200-native hiccup encode/decode hot path.
 *
 * The reference (nhomble/hiccup) has no FFI: its boundary is the Python function API of
 * hiccup/compression.py and hiccup/codec.py.  Each entry point below names the reference code it
 * replaces (file:line under /root/reference); hiccup_b200/compression.py and hiccup_b200/codec.py
 * compose them back into the reference's eight functions, and INTEGRATION.md shows the ctypes
 * binding a maintainer of the reference would add.
 *
 * Conventions
 *   - every function returns 0 on success, a negative hic_status on failure;
 *     hic_last_error() returns the message of the calling thread's last failure;
 *   - all pointers are caller-owned; `d_` arguments are device pointers on the current CUDA device,
 *     `h_` arguments are host pointers; `stream` is a cudaStream_t passed as void* (NULL = default);
 *   - calls are asynchronous on `stream` unless the comment says otherwise; no hidden global state
 *     besides read-only constant tables;
 *   - images are H x W x 3 uint8, C-contiguous, channel 0 treated as R (the reference feeds BGR
 *     from cv2.imread through the same arithmetic, run.py:19);
 *   - batches are n images of one shape, contiguous.
 *
 * Coefficient layout ("zigzag blocks"): per image, luminance blocks, then Cr blocks, then Cb
 * blocks; blocks in raster block order of their (zero-padded) plane; each block is 64 int16 in the
 * reference's scan order (transform._zigzag_indices, transform.py:106-124), i.e. one 128-byte line.
 * Coefficients that fall outside the unpadded plane are zero, as they are after the reference's
 * crop (transform.py:63) and re-pad (codec.py:288,294).
 */
#ifndef HICCUP_B200_H
#define HICCUP_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum hic_status {
    HIC_OK = 0,
    HIC_ERR_INVALID = -1,     /* bad argument */
    HIC_ERR_CUDA = -2,        /* CUDA runtime error; message has the details */
    HIC_ERR_CAPACITY = -3,    /* an output buffer was too small; nothing past its end was written */
    HIC_ERR_CORRUPT = -4      /* a bit stream did not decode to the expected symbol count */
} hic_status;

/* ---- runtime plumbing ------------------------------------------------------------------------ */
int hic_version(void);
const char* hic_last_error(void);
int hic_device_count(int* count);
int hic_set_device(int device);
int hic_get_device(int* device);          /* the calling thread's current CUDA device */
/* How host threads wait for the current device from now on: 1 = block (yield the core), 0 = the driver's
 * default (spin when cores are plentiful).  Optional: PipelinedCodec(blocking_sync=True) uses it for its
 * per-slot host threads; on the boxes measured spinning was faster (batch.py). */
int hic_set_blocking_sync(int on);
int hic_device_name(char* buf, size_t buflen);
int hic_malloc(void** d_ptr, size_t bytes);
int hic_free(void* d_ptr);
int hic_host_alloc(void** h_ptr, size_t bytes);          /* pinned */
int hic_host_free(void* h_ptr);
/* Page-lock host memory the caller already owns (e.g. a /dev/shm mapping several ranks of one box share)
 * so that bulk copies to and from it run asynchronously at full PCIe rate; portable across contexts.
 * The reference is one process on one image (run.py:18-43); these two and hic_ticket_take exist for the
 * box-wide job queue of hiccup_b200/jobs.py (by-image partition with link-aware load balancing). */
int hic_host_register(void* h_ptr, size_t bytes);
int hic_host_unregister(void* h_ptr);
/* Atomically take `count` tickets from a 64-bit counter in (possibly shared, process-crossing) host
 * memory: *first = the old value, counter += count.  h_counter must be 8-byte aligned. */
int hic_ticket_take(void* h_counter, int64_t count, int64_t* first);
int hic_memcpy_h2d(void* d_dst, const void* h_src, size_t bytes, void* stream);
int hic_memcpy_d2h(void* h_dst, const void* d_src, size_t bytes, void* stream);
int hic_memset(void* d_ptr, int value, size_t bytes, void* stream);
int hic_stream_create(void** stream);
int hic_stream_destroy(void* stream);
int hic_stream_sync(void* stream);                       /* blocks the host */

/* Per-kernel timing with CUDA events recorded on the launching stream around every kernel this
 * library launches.  hic_profile_report synchronises, writes {"kernel": [total_ms, launches], ...}
 * as JSON into buf and clears the record. */
int hic_profile_enable(int on);
int hic_profile_report(char* buf, size_t buflen);
/* The spans recorded so far as a JSON array of [kernel, stream number, start ms, end ms] (relative to the
 * first span); does not clear them.  A development aid for pipelined runs over several CUDA streams. */
int hic_profile_timeline(char* buf, size_t buflen);

/* ---- DCT-mode geometry ----------------------------------------------------------------------- */
typedef struct hic_dct_geometry {
    int32_t h, w;             /* luminance plane = image */
    int32_t hc, wc;           /* chroma planes after pyrDown: h/2, w/2 (transform.py:160-166) */
    int32_t nby_l, nbx_l;     /* luminance blocks: ceil(h/8), ceil(w/8) (transform.py:17-42) */
    int32_t nby_c, nbx_c;     /* chroma blocks */
    int64_t nb_l, nb_c;       /* blocks per plane */
    int64_t blocks_per_image; /* nb_l + 2 nb_c */
    int32_t out_h, out_w;     /* decoded image: 2 hc, 2 wc (transform.force_merge, :269-277) */
} hic_dct_geometry;
int hic_dct_geometry_of(int32_t h, int32_t w, hic_dct_geometry* out);

/* One rounding-tie candidate: a block whose float32 quantised value landed inside the error band
 * around a half-integer at one or more scan positions (bit k of mask = scan position k). */
typedef struct hic_tie_record {
    uint32_t block;           /* global block index: image * blocks_per_image + block in image */
    uint32_t reserved;
    uint64_t mask;
} hic_tie_record;

/* d_stats[0] candidates flagged (blocks), [1] coefficients re-evaluated in float64,
 * [2] coefficients whose float32 rounding was changed by the re-evaluation, [3] records dropped
 * because tie_capacity was too small (if non-zero the coefficients are NOT guaranteed exact). */
#define HIC_TIE_STATS 4

/* K1 -- fused encode transform.  Replaces compression.jpeg_compression (compression.py:16-39):
 * cv2.cvtColor RGB->YCrCb, cv2.pyrDown of both chroma planes, x-128, zero pad, 8x8 DCT-II
 * (scipy.fftpack.dct rows then columns), division by the Annex-K table, np.round, crop; plus the
 * zigzag of transform.ac_components (transform.py:260-266).  float32 butterflies; every value
 * within the float32 error band of a rounding tie is then re-evaluated by a second kernel in
 * float64 with scipy's exact operation order, so the output equals the reference's bit for bit.
 * d_ties needs room for tie_capacity records -- hic_dct_tie_capacity() gives the count that is
 * always enough: one record per block plus the per-warp flag words K1 leaves at the buffer's tail;
 * d_coef must be 128-byte aligned (its blocks leave through TMA tensor stores);
 * d_stats is HIC_TIE_STATS uint32, zeroed by this call. */
int hic_dct_tie_capacity(int32_t n, int32_t h, int32_t w, uint32_t* out);
int hic_dct_forward(const uint8_t* d_rgb, int32_t n, int32_t h, int32_t w, int16_t* d_coef,
                    hic_tie_record* d_ties, uint32_t tie_capacity, uint32_t* d_stats, void* stream);

/* Zigzag blocks <-> the reference's CompressedImage planes (model.py:38-74): int32, cropped to the
 * unpadded plane shape, block (by,bx) coefficient (u,v) at [8by+u, 8bx+v] (transform.py:45-64). */
int hic_blocks_to_planes(const int16_t* d_coef, int32_t n, int32_t h, int32_t w, int32_t* d_lum,
                         int32_t* d_cr, int32_t* d_cb, void* stream);
int hic_planes_to_blocks(const int32_t* d_lum, const int32_t* d_cr, const int32_t* d_cb, int32_t n,
                         int32_t h, int32_t w, int16_t* d_coef, void* stream);

/* K7+K8 -- decode transform.  Replaces compression.jpeg_decompression (compression.py:42-56):
 * coefficient * table, idct rows then columns, /256, +128, astype(uint8) (truncate, wrap),
 * cv2.pyrUp of both chroma planes, crop of the luminance plane, cv2.cvtColor YCrCb->RGB.
 * d_y (n*h*w), d_cr, d_cb (n*hc*wc each) are scratch planes; d_rgb_out is n*out_h*out_w*3.
 * float32 butterflies; every sample within the float32 error band of an integer (where the
 * reference's uint8 truncation steps) is re-evaluated in float64 with scipy's exact operation
 * order before the (integer) upsampling and colour conversion, so pixels equal the reference's.
 * d_ties / tie_capacity / d_stats as for hic_dct_forward (mask bit i = sample 8*y + x). */
int hic_dct_inverse(const int16_t* d_coef, int32_t n, int32_t h, int32_t w, uint8_t* d_y,
                    uint8_t* d_cr, uint8_t* d_cb, uint8_t* d_rgb_out, hic_tie_record* d_ties,
                    uint32_t tie_capacity, uint32_t* d_stats, void* stream);

/* Thumbnail -- a 1/8-scale preview from the DC terms alone: one pixel per 8x8 tile of the image
 * compression.jpeg_decompression (compression.py:42-56) returns, th = ceil(out_h / 8) rows of tw =
 * ceil(out_w / 8).  Each block counts as its DC-only decode through transform.inv_dct_channel
 * (transform.py:169-179), the constant ((q T00 + 32768) / 256 truncated toward zero) & 255 (T00 = 16
 * luminance, 17 chroma); the chroma planes of those values go through cv2.pyrUp (transform.py:151-157),
 * all three are cropped to th x tw and converted by cv2.cvtColor YCrCb->RGB (compression.py:56), the
 * integer arithmetic of K8.  d_dc: one int16 DC value per block in global block order (image *
 * blocks_per_image + block), as hic_decode_run_dc leaves them; d_rgb_out: n * th * tw * 3.
 * hic_dct_thumbnail_shape is host only (no device needed). */
int hic_dct_thumbnail_shape(int32_t h, int32_t w, int32_t* th, int32_t* tw);
int hic_dct_thumbnail(const int16_t* d_dc, int32_t n, int32_t h, int32_t w, uint8_t* d_rgb_out, void* stream);

/* Region -- one rh x rw window of the decoded image per image of the batch, at full resolution:
 * window i equals compression.jpeg_decompression(...)[top:top+rh, left:left+rw] (compression.py:42-56)
 * bit for bit, (top, left) = h_origin[2i], h_origin[2i+1] in output coordinates; valid when top, left >= 0,
 * rh, rw >= 1, top + rh <= out_h and left + rw <= out_w.  Output pixel (oy, ox) reads luminance sample
 * (oy, ox) and the chroma samples of rows {ym, cy, yn} and columns {xm, cx, xn}, cy = oy >> 1, cx = ox >> 1,
 * ym = cy > 0 ? cy - 1 : (hc > 1 ? 1 : 0), yn = min(cy + 1, hc - 1) (the same for columns): cv2.pyrUp's
 * borders at the image's edges (reflect at the top and left, replicate at the bottom and right), the real
 * neighbouring samples everywhere else.  Only the blocks covering those samples are inverse-transformed
 * (K7's float32 path, its error band and float64 fix-up; tie records carry the global block index) into
 * window-local 8x8 tiles in d_work, and only the window's pixels are upsampled and converted (K8's integer
 * arithmetic) straight into d_rgb_out (n * rh * rw * 3).
 * hic_dct_region_blocks (host only) gives the block rectangles a window at (top, left) selects:
 * rect = {by, bx, nby, nbx} of the luminance plane, then the same of each chroma plane; every window of one
 * size selects rectangles of one size.  hic_dct_region_sizes (host only) gives the d_work bytes and the tie
 * capacity (one record per selected block) for n windows of rh x rw.  hic_dct_region checks every origin on
 * the host (HIC_ERR_INVALID for a window outside out_h x out_w or an empty size) before anything is launched,
 * and copies the origins to d_work with cudaMemcpyAsync on `stream`.  d_coef as hic_dct_inverse reads it
 * (16-byte aligned); d_work 16-byte aligned; d_stats as for hic_dct_inverse, zeroed by this call. */
int hic_dct_region_blocks(int32_t h, int32_t w, int32_t top, int32_t left, int32_t rh, int32_t rw, int32_t* rect);
int hic_dct_region_sizes(int32_t n, int32_t h, int32_t w, int32_t rh, int32_t rw, size_t* work_bytes,
                         uint32_t* tie_capacity);
int hic_dct_region(const int16_t* d_coef, int32_t n, int32_t h, int32_t w, const int32_t* h_origin,
                   int32_t rh, int32_t rw, uint8_t* d_work, size_t work_bytes, hic_tie_record* d_ties,
                   uint32_t tie_capacity, uint32_t* d_stats, uint8_t* d_rgb_out, void* stream);

/* Scaled decode -- the 1/s-scale image of each image of the batch, s = scale = 2 or 4 (scale 8 is
 * hic_dct_thumbnail), m = 8 / s samples per block side.  Every block of the zero-padded planes gives an
 * m x m tile: X = q T (u, v < m; the block's other coefficients are ignored), A = X B^T (rows first), Y = B A,
 * each sum left to right in float64 with every product and sum rounded, sample = (uint8)(Y / 256 + 128)
 * (truncation toward zero, wrap).  B_s[k][0] = 1, B_s[k][n] = 2 D(n) cos(pi n (2k+1) / (2m)),
 * D(n) = sin(pi n s / 16) / (s sin(pi n / 16)) (hex literals in csrc/hic_core.cuh): B X B^T is the mean of each
 * s x s tile of the unrounded 8 x 8 IDCT of a block with no coefficients beyond u, v < m.  The tiles form
 * Y_s (m nby_l x m nbx_l) and Cr_s, Cb_s (m nby_c x m nbx_c); Cr_s and Cb_s go through cv2.pyrUp's integer
 * rules, and all three are cropped to sh x sw = ceil(out_h / s) x ceil(out_w / s) and converted by
 * ycrcb_to_rgb into d_rgb_out (n * sh * sw * 3) -- the thumbnail's convention, which is this definition at
 * m = 1.  The coefficients come from K7's buffer (d_coef, 16-byte aligned), only the first 64 (s = 2) or 16
 * (s = 4) bytes of each block; a float32 transform with a rigorous error band, whose flagged blocks are
 * re-evaluated in float64 (tie records carry the global block index), writes the tiles to d_work
 * (16-byte aligned).  hic_dct_scaled_shape and hic_dct_scaled_sizes (host only) give sh x sw and the d_work
 * bytes and tie capacity (one record per block).  Every entry point returns HIC_ERR_INVALID for a scale other
 * than 2 or 4 before anything is launched.  d_stats as for hic_dct_inverse, zeroed by this call; [1] counts
 * samples re-evaluated. */
int hic_dct_scaled_shape(int32_t h, int32_t w, int32_t scale, int32_t* sh, int32_t* sw);
int hic_dct_scaled_sizes(int32_t n, int32_t h, int32_t w, int32_t scale, size_t* work_bytes, uint32_t* tie_capacity);
int hic_dct_scaled(const int16_t* d_coef, int32_t n, int32_t h, int32_t w, int32_t scale, uint8_t* d_work,
                   size_t work_bytes, hic_tie_record* d_ties, uint32_t tie_capacity, uint32_t* d_stats,
                   uint8_t* d_rgb_out, void* stream);

/* Scaled region -- one rh x rw window of the 1/s-scale image per image of the batch: window i equals
 * hic_dct_scaled's image (s = 2, 4) or hic_dct_thumbnail's (s = 8) cropped to [top, top+rh) x [left, left+rw)
 * bit for bit, (top, left) = h_origin[2i], h_origin[2i+1] in the coordinates of that sh x sw = ceil(out_h / s) x
 * ceil(out_w / s) image; valid when top, left >= 0, rh, rw >= 1, top + rh <= sh and left + rw <= sw.
 * hic_dct_scaled_region (s = 2, 4) selects blocks with the region rules at m = 8 / s samples per block side: the
 * window reads rows [top, top+rh) of the reduced luminance plane and the pyrUp taps of the reduced chroma planes
 * (m nby_c x m nbx_c, hic_dct_scaled's borders).  Only those blocks go through hic_dct_scaled's float32 transform,
 * its error band and float64 fix-up (tie records carry the global block index) into window-local tiles in d_work,
 * and only the window's pixels are upsampled and converted, straight into d_rgb_out (n * rh * rw * 3).  d_coef as
 * hic_dct_scaled reads it (16-byte aligned; only the first 64 (s = 2) or 16 (s = 4) bytes of a selected block);
 * d_work 16-byte aligned; d_stats as for hic_dct_scaled, zeroed by this call.
 * hic_dct_thumbnail_region computes the 1/8-scale window's pixels straight from the DC values d_dc (as
 * hic_dct_thumbnail reads them, 2-byte aligned); d_work (4-byte aligned) needs 8 n bytes, for the origins.
 * Both check every origin on the host (HIC_ERR_INVALID for a window outside sh x sw or an empty size) before
 * anything is launched and copy the origins to d_work with cudaMemcpyAsync on `stream`.
 * hic_dct_scaled_region_blocks (host only, s = 2, 4) gives the block rectangles a window selects, as
 * hic_dct_region_blocks does; every window of one size selects rectangles of one size.
 * hic_dct_scaled_region_sizes (host only, s = 2, 4, 8) gives the d_work bytes and the tie capacity (one record per
 * selected block; 0 at s = 8) for n windows of rh x rw.  hic_dct_scaled_region returns HIC_ERR_INVALID for a scale
 * other than 2 or 4 before anything is launched. */
int hic_dct_scaled_region_blocks(int32_t h, int32_t w, int32_t scale, int32_t top, int32_t left, int32_t rh, int32_t rw,
                                 int32_t* rect);
int hic_dct_scaled_region_sizes(int32_t n, int32_t h, int32_t w, int32_t scale, int32_t rh, int32_t rw,
                                size_t* work_bytes, uint32_t* tie_capacity);
int hic_dct_scaled_region(const int16_t* d_coef, int32_t n, int32_t h, int32_t w, int32_t scale, const int32_t* h_origin,
                          int32_t rh, int32_t rw, uint8_t* d_work, size_t work_bytes, hic_tie_record* d_ties,
                          uint32_t tie_capacity, uint32_t* d_stats, uint8_t* d_rgb_out, void* stream);
int hic_dct_thumbnail_region(const int16_t* d_dc, int32_t n, int32_t h, int32_t w, const int32_t* h_origin,
                             int32_t rh, int32_t rw, uint8_t* d_work, size_t work_bytes, uint8_t* d_rgb_out, void* stream);

/* ---- wavelet ("HIC") mode --------------------------------------------------------------------- */
/* Sub-band geometry of pywt.wavedec2(channel, "db1", level=3) (transform.py:196-209): level sizes
 * ceil(n / 2) per level; ten sub-bands per channel in the order [cA3, cH3, cV3, cD3, cH2, cV2, cD2,
 * cH1, cV1, cD1]; band_off[b] = first element of band b in the channel's concatenated stream. */
typedef struct hic_wavelet_geometry {
    int32_t h, w;
    int32_t lh[4], lw[4];     /* [0] = image, [l] = sub-band shape at level l */
    int64_t band_off[10];
    int64_t len;              /* coefficients per channel */
} hic_wavelet_geometry;
int hic_wavelet_geometry_of(int32_t h, int32_t w, hic_wavelet_geometry* out);

/* K9 -- fused wavelet encode transform.  Replaces compression.wavelet_compression
 * (compression.py:59-85: cvtColor, x - 256, pywt.wavedec2 db1 level 3, subband_quantize
 * (quantization.py:60-69: cA rounded, detail level i = 0 (coarsest) .. 2 divided by i*i + 1, np.round),
 * threshold |v| < 5 -> 0 (transform.py:227-239)) plus the zigzag of every whole sub-band and their
 * concatenation (codec.wavelet_encode, codec.py:123-126).  float64, PyWavelets' operation order.
 * d_flat: the flat-mode stream of hic_layout_flat(n, geometry.len): channel stream (image, c) starts at
 * element 64 * ceil(len / 64) * (3 image + c). */
int hic_wavelet_forward(const uint8_t* d_rgb, int32_t n, int32_t h, int32_t w, int16_t* d_flat, void* stream);
/* K10 -- fused wavelet decode transform.  Replaces codec.wavelet_decode_pull_subbands (codec.py:166-179)
 * and compression.wavelet_decompression (compression.py:88-100).  h and w must be multiples of 8 (the
 * reference's decoder assumes exact doubling between levels, codec.py:182-189). */
int hic_wavelet_inverse(const int16_t* d_flat, int32_t n, int32_t h, int32_t w, uint8_t* d_rgb_out, void* stream);
/* Flat stream <-> the reference's CompressedImage sub-bands (model.py:38-74): per image and channel the
 * ten raster int32 sub-bands concatenated in band order (geometry.len values). */
int hic_wavelet_flat_to_bands(const int16_t* d_flat, int32_t n, int32_t h, int32_t w, int32_t* d_bands, void* stream);
int hic_wavelet_bands_to_flat(const int32_t* d_bands, int32_t n, int32_t h, int32_t w, int16_t* d_flat, void* stream);

/* Wavelet mode at settings other than the defaults (reference settings.py:12-16): WAVELET_NUM_LEVELS in
 * 1..HIC_WAVELET_MAX_LEVELS, any non-zero WAVELET_SUBBAND_QUANTIZATION_MULTIPLIER, any WAVELET_THRESHOLD,
 * and WAVELET_QUALITY_FACTOR < 1 -- the order statistic of quantization.quality_threshold_value
 * (quantization.py:84-94) over all coefficients of a channel, taken on the device from a 65536-bin
 * histogram.  db1 / haar only (model.py:31-35).  Same arithmetic as K9 / K10, level by level. */
#define HIC_WAVELET_MAX_LEVELS 5
typedef struct hic_wavelet_params {
    int32_t levels;            /* settings.WAVELET_NUM_LEVELS */
    int32_t reserved;
    double multiplier;         /* settings.WAVELET_SUBBAND_QUANTIZATION_MULTIPLIER (!= 0) */
    double threshold;          /* settings.WAVELET_THRESHOLD (0: none) */
    int64_t threshold_index;   /* len - ceil(len * WAVELET_QUALITY_FACTOR), or -1 for a quality factor of 1 */
} hic_wavelet_params;
typedef struct hic_wavelet_pyramid {
    int32_t h, w, levels, n_bands;     /* n_bands = 3 levels + 1: [cA_L, (cH, cV, cD)_L, ..., (cH, cV, cD)_1] */
    int32_t lh[6], lw[6];              /* [0] = image, [l] = sub-band shape at level l */
    int64_t band_off[16];
    int64_t len;                       /* coefficients per channel */
} hic_wavelet_pyramid;
int hic_wavelet_pyramid_of(int32_t h, int32_t w, int32_t levels, hic_wavelet_pyramid* out);
/* bytes of device scratch the two transforms below need (float64 planes of the running approximation) */
int hic_wavelet_general_work_bytes(int32_t n, int32_t h, int32_t w, size_t* out);
/* compression.wavelet_compression (compression.py:59-85) + the sub-band zigzag of codec.wavelet_encode
 * (codec.py:123-126); d_flat as for hic_wavelet_forward with len = pyramid.len */
int hic_wavelet_forward_general(const uint8_t* d_rgb, int32_t n, int32_t h, int32_t w, const hic_wavelet_params* params,
                                void* d_work, int16_t* d_flat, void* stream);
/* compression.wavelet_decompression (compression.py:88-100).  h and w: the even sides 2 lh[1], 2 lw[1] of the
 * image pywt.waverec2 returns (it trims the extra row / column between levels of odd size) */
int hic_wavelet_inverse_general(const int16_t* d_flat, int32_t n, int32_t h, int32_t w, const hic_wavelet_params* params,
                                void* d_work, uint8_t* d_rgb_out, void* stream);
/* Scaled decode -- the 1/s-scale image of a wavelet file of L = params->levels levels, s = 2^k with
 * 1 <= k <= L, h and w multiples of 2^L: (h / s) x (w / s) x 3 per image into d_rgb_out.  Per channel:
 * dequantise as compression.wavelet_decompression does (A_L = cA_L; detail group i, 0 = coarsest, times
 * params->multiplier * (i*i + 1); the thresholds are not used); A_k is the running approximation after the
 * first L - k reconstruction levels of waverec2 -- the same operations in the same order as
 * hic_wavelet_inverse_general, so bit for bit the intermediate it holds (at k = L, cA_L itself);
 * sample = astype(uint8)(A_k * 2^-k + 256) (the product is exact; truncation toward zero, wrap).  The three
 * reduced planes go through ycrcb_to_rgb (no chroma subsampling, no crop).  For db1, A_k * 2^-k is the mean
 * of each s x s tile of the unrounded full reconstruction.  Only cA_L and the detail bands of levels
 * L .. k + 1 are read.  d_work: hic_wavelet_general_work_bytes(n, h, w).  Returns HIC_ERR_INVALID for a bad
 * scale or shape before anything is launched.  This is also the path at the default settings: a fused
 * K10-style kernel measured slower on a B200 (DESIGN.md section 6). */
int hic_wavelet_scaled_general(const int16_t* d_flat, int32_t n, int32_t h, int32_t w, const hic_wavelet_params* params,
                               int32_t scale, void* d_work, uint8_t* d_rgb_out, void* stream);
/* Region -- one rh x rw window of the full-resolution (s = 1) or 1/s-scale image per image of the batch,
 * s = 2^k with 0 <= k <= L = params->levels, h and w multiples of 2^L: window i equals
 * hic_wavelet_inverse_general's image (s = 1; K10's at the defaults) or hic_wavelet_scaled_general's (s >= 2)
 * cropped to [top, top+rh) x [left, left+rw) bit for bit, (top, left) = h_origin[2i], h_origin[2i+1] in the
 * coordinates of that (h / s) x (w / s) image; valid when top, left >= 0, rh, rw >= 1, top + rh <= h / s and
 * left + rw <= w / s.  The arithmetic is at params->levels and params->multiplier; the thresholds are not used.
 * db1 has no halo, so at each level l > k only the window's dyadic parent rectangle, rows
 * [top >> (l - k), (top + rh - 1) >> (l - k)] and the same for columns, of cA_L and of the detail bands is read,
 * and each sample on that path is computed with the full inverse's operations in its order, straight into
 * d_rgb_out (n * rh * rw * 3): no float64 planes.  d_work (4-byte aligned) needs 8 n bytes, for the origins,
 * which are copied there with cudaMemcpyAsync on `stream`.  Returns HIC_ERR_INVALID for a scale other than 2^k,
 * 0 <= k <= L, sides that are not multiples of 2^L, an empty size, a window outside (h / s) x (w / s) or
 * work_bytes < 8 n, all checked on the host before anything is launched. */
int hic_wavelet_region(const int16_t* d_flat, int32_t n, int32_t h, int32_t w, const hic_wavelet_params* params,
                       int32_t scale, const int32_t* h_origin, int32_t rh, int32_t rw, void* d_work, size_t work_bytes,
                       uint8_t* d_rgb_out, void* stream);
int hic_wavelet_flat_to_bands_general(const int16_t* d_flat, int32_t n, int32_t h, int32_t w, int32_t levels, int32_t* d_bands,
                                      void* stream);
int hic_wavelet_bands_to_flat_general(const int32_t* d_bands, int32_t n, int32_t h, int32_t w, int32_t levels, int16_t* d_flat,
                                      void* stream);

/* ---- entropy stage ---------------------------------------------------------------------------- */
/* A batch is 3 n "channel streams" (image i, channel c in lum, cr, cb).  Each channel stream is a
 * run of 64-element int16 blocks.  DCT mode (skip_first = 1): element 0 of every block is its DC
 * term and the AC stream is elements 1..63 of all blocks in order (transform.ac_components,
 * transform.py:260-266).  Flat mode (skip_first = 0, wavelet): the stream is simply the first
 * len[c] elements (the ten zigzagged sub-bands concatenated, codec.py:123-126).
 * Every channel stream yields symbol streams, indexed  s = (image * 3 + channel) * 3 + kind:
 * kind 0 = DC differences (DCT mode only), 1 = run-length values, 2 = run-length zero counts. */
typedef struct hic_stream_layout {
    int32_t n_images;
    int32_t skip_first;
    int64_t blocks_per_image;
    int64_t nb[3];            /* blocks per channel stream */
    int64_t block_off[3];     /* first block of channel c inside an image */
    int64_t len[3];           /* run-length input positions per channel stream */
} hic_stream_layout;
int hic_layout_dct(int32_t n, int32_t h, int32_t w, hic_stream_layout* out);
int hic_layout_flat(int32_t n, int64_t len, hic_stream_layout* out);   /* blocks = ceil(len/64), same for all 3 */

#define HIC_KIND_DC 0
#define HIC_KIND_VALUE 1
#define HIC_KIND_LENGTH 2

typedef struct hic_entropy_plan hic_entropy_plan;      /* owns the device workspace of one batch shape */

/* value_bins: power of two; symbols must lie in [-value_bins/2, value_bins/2).  8192 covers every
 * value K1 / the wavelet kernels can produce; 65536 covers all of int16. */
int hic_entropy_plan_create(const hic_stream_layout* layout, int32_t value_bins, hic_entropy_plan** out);
int hic_entropy_plan_destroy(hic_entropy_plan* plan);

/* E1 (device) -- DC differences (codec.differential_coding, codec.py:47-52; utils.differences,
 * utils.py:51-63), run-length symbols (codec.run_length_coding, codec.py:55-99: symbol = (zeros
 * before, value); a run l >= 15 becomes l/15 fillers (14, 0) then (l mod 15, value); trailing
 * zeros collapse to one (0, 0)), and per-stream symbol histograms with first-occurrence indices
 * (utils.group_by, utils.py:83-96, via huffman.py:17-19). */
int hic_entropy_symbolize(hic_entropy_plan* plan, const int16_t* d_coef, void* stream);

/* ---- row-band sharding of one tall image (SURVEY 8(e)): E1 in two passes with the seam state in
 * between, externally built codes, raw bit strings at a bit phase ------------------------------ */
/* What crosses a band seam for one channel stream (index image * 3 + channel). */
typedef struct hic_band_carry {
    int32_t carry_zeros;      /* zero positions since the last non-zero of the bands above (0 for the top band) */
    int32_t prev_dc;          /* DC value of the last block of the band above (0 for the top band) */
    int32_t more_after;       /* a band below still holds a non-zero: trailing zeros here keep emitting fillers */
    int32_t closes_stream;    /* bottom band: append the (0, 0) if the whole stream ends in zeros */
} hic_band_carry;
/* Pass 1: per-tile run summaries; h_first_nz / h_last_nz (3 n entries) receive the first and last
 * non-zero run-length position of every channel stream (-1: none).  Synchronises `stream`. */
int hic_entropy_scan(hic_entropy_plan* plan, const int16_t* d_coef, int32_t* h_first_nz, int32_t* h_last_nz, void* stream);
/* Pass 2 (after hic_entropy_scan): symbols, DC differences and histograms with the seam state applied,
 * so that the band's symbol lists are exactly its slice of the whole image's lists (codec.py:47-99
 * runs over the whole channel).  h_band: 3 n entries, or NULL for stand-alone streams.
 * hic_entropy_symbolize = scan + emit(NULL). */
int hic_entropy_emit(hic_entropy_plan* plan, const int16_t* d_coef, const hic_band_carry* h_band, void* stream);
/* The compacted histograms of the last emit: h_index[2 s], h_index[2 s + 1] = first entry and entry
 * count of symbol stream s; h_entries: (symbol, count, first occurrence index) int32 triples;
 * h_nsym_rl (3 n entries, may be NULL): run-length symbols per channel stream.  Synchronises. */
int hic_entropy_histograms(hic_entropy_plan* plan, uint32_t* h_index, int32_t* h_entries, uint64_t capacity,
                           uint64_t* n_entries, uint32_t* h_nsym_rl, void* stream);
/* Install codes built elsewhere (the merged tables of all bands) in the packed layout of
 * hic_entropy_tables_packed, with the symbol and bit counts of THIS plan's streams.  h_start_bit[s]:
 * 8 (or NULL) = framed payload as usual; 0..7 = hic_entropy_pack writes the raw bits of stream s
 * starting at that bit of its first byte, no pad-count byte (the host ORs the band strings together).
 * Synchronises `stream`. */
int hic_entropy_set_codes(hic_entropy_plan* plan, const uint32_t* h_index, const int32_t* h_row_sym,
                          const uint64_t* h_row_packed, uint64_t total_rows, const uint32_t* h_nsym,
                          const uint64_t* h_nbits, const uint32_t* h_start_bit, void* stream);

/* E2 (host; synchronises `stream`) -- fetch the compacted histograms, build every Huffman code
 * exactly as HuffmanTree._construct does (huffman.py:60-79, heapq replay), upload code tables. */
int hic_entropy_build_codes(hic_entropy_plan* plan, void* stream);

/* E2 on the device -- the same heapq replay, one lane per symbol stream with its heap in shared
 * memory (alphabets up to 8192 symbols); nothing but 32 bytes of totals crosses PCIe.  Produces
 * exactly the codes of hic_entropy_build_codes (tests/test_gpu_codec.py compares them).  The
 * per-stream results and tables are downloaded lazily by the two query functions below.
 * Once a plan has built its codes here, its next hic_entropy_symbolize / hic_entropy_emit launches
 * the DC streams' pass itself, on the plan's own CUDA streams beside the run-length kernels (the
 * other builders wait for it); results do not depend on that.  With HIC_ENTROPY_SERIAL set in the
 * environment everything stays on `stream`, one kernel after the other (per-kernel timing). */
int hic_entropy_build_codes_device(hic_entropy_plan* plan, void* stream);

/* Results of E2, all host arrays indexed by symbol stream s (9 n entries; kind 0 entries are
 * empty in flat mode).  rows[s]: table rows; nsym[s]: symbols; nbits[s]: Huffman-coded bits;
 * byte_off[s] / byte_len[s]: where hic_entropy_pack puts the framed bytes of stream s. */
int hic_entropy_stream_info(hic_entropy_plan* plan, uint32_t* h_rows, uint32_t* h_nsym, uint64_t* h_nbits,
                            uint64_t* h_byte_off, uint64_t* h_byte_len, uint64_t* total_rows, uint64_t* total_bytes);
/* Table rows of all streams concatenated in s order, each stream's rows in first-occurrence order
 * (what HuffmanTree.encode_table returns, huffman.py:144-147): symbol, code length, code bits
 * (right aligned; first bit of the code string = most significant; '1' = left = first popped). */
int hic_entropy_tables(hic_entropy_plan* plan, int32_t* h_symbols, uint8_t* h_lens, uint64_t* h_codes);

/* The same tables without any host-side reshaping, for the batched path: the rows exactly as they
 * sit on the device (each stream's rows contiguous and in first-occurrence order, streams in no
 * particular order), rows packed as (length << 58 | code bits), and h_index[2 s], h_index[2 s + 1] =
 * first row and row count of stream s.  Asynchronous device-to-host copies on `stream` into the
 * caller's (ideally pinned) arrays of hic_entropy_stream_info's total_rows entries; synchronise
 * `stream` before reading them. */
int hic_entropy_tables_packed(hic_entropy_plan* plan, uint32_t* h_index, int32_t* h_row_sym, uint64_t* h_row_packed,
                              void* stream);

/* E3 (device) -- concatenate the codes of every symbol stream (HuffmanTree.encode_data,
 * huffman.py:131-142) and frame them as iohelper.padded_bs_2_bytes does (iohelper.py:35-48):
 * byte 0 = p = 8 - (nbits mod 8), then the bits MSB first, then p zero bits.  d_out must hold
 * total_bytes; it is zeroed by the call. */
int hic_entropy_pack(hic_entropy_plan* plan, uint8_t* d_out, void* stream);

/* Device-resident code tables of the last build (either flavour), for handing straight to
 * hic_decode_set_tables_device: per-stream {uint32 offset, uint32 count} index, row symbols, and
 * rows packed as (length << 58 | code bits). */
int hic_entropy_device_tables(const hic_entropy_plan* plan, const void** d_index, const int32_t** d_row_sym,
                              const uint64_t** d_row_packed, const uint64_t** d_byte_off, const uint64_t** d_nbits);

/* The host Huffman construction on its own (no CUDA call): leaf frequencies in first-occurrence
 * order -> code length and bits per leaf.  Replaces HuffmanTree._construct + encode_table
 * (huffman.py:60-79, 144-147).  Returns HIC_ERR_INVALID if a code would exceed 58 bits. */
int hic_huffman_build_host(const uint32_t* h_freqs, uint32_t n, uint8_t* h_lens, uint64_t* h_codes);

/* Device pointers into the plan's workspace (valid until the plan is destroyed), for tests and
 * for the band-sharded path: DC differences (int16, indexed by global block), run-length values
 * (int16) and zero counts (uint8) (channel stream cs starts at 64 * first block of cs). */
int hic_entropy_symbol_buffers(const hic_entropy_plan* plan, const int16_t** d_dc, const int16_t** d_values,
                               const uint8_t** d_lengths);

/* ---- entropy decode --------------------------------------------------------------------------- */
typedef struct hic_decode_plan hic_decode_plan;
int hic_decode_plan_create(const hic_stream_layout* layout, hic_decode_plan** out);
int hic_decode_plan_destroy(hic_decode_plan* plan);
/* Code tables of every symbol stream (same layout as hic_entropy_tables) -- replaces
 * HuffmanTree.construct_from_coding (huffman.py:30-58). */
int hic_decode_set_tables(hic_decode_plan* plan, const uint32_t* h_rows, const int32_t* h_symbols,
                          const uint8_t* h_lens, const uint64_t* h_codes, void* stream);
/* The same from the packed host layout of hic_entropy_tables_packed.  Asynchronous: the host arrays
 * must stay valid until `stream` has been synchronised. */
int hic_decode_set_tables_packed(hic_decode_plan* plan, const uint32_t* h_index, const int32_t* h_row_sym,
                                 const uint64_t* h_row_packed, uint64_t total_rows, void* stream);
/* The same from device-resident tables (hic_entropy_device_tables); the arrays are referenced, not
 * copied, and must stay valid until decoding is done.  total_rows: an upper bound on first row + row
 * count over the streams (hic_entropy_stream_info's total_rows).  Asynchronous. */
int hic_decode_set_tables_device(hic_decode_plan* plan, const void* d_index, const int32_t* d_row_sym,
                                 const uint64_t* d_row_packed, uint64_t total_rows, void* stream);
/* D1-D3 (device) -- Huffman decode (HuffmanTree.decode_data, huffman.py:149-174), run-length
 * expansion (codec.decode_run_length, codec.py:102-113), DC prefix sum (utils.invert_differences,
 * utils.py:66-74) and de-zigzag into blocks (codec.py:415-425).  d_bytes holds the framed byte
 * strings (each 4-byte aligned at h_byte_off[s], with 8 readable bytes after the last one);
 * h_nbits[s] is the payload bit count of stream s (8 * (framed length - 1) - pad count, 0 for an
 * absent stream).  d_coef receives zigzag blocks.  Synchronises `stream` and returns
 * HIC_ERR_CORRUPT if a stream decodes to the wrong length. */
/* The C ABI takes d_bytes without a length; a caller that knows it says so here and every later run checks that
 * each stream's words lie inside the buffer (0 = unknown again).  Returns HIC_ERR_INVALID from the run otherwise. */
int hic_decode_set_data_bytes(hic_decode_plan* plan, uint64_t nbytes);
int hic_decode_run(hic_decode_plan* plan, const uint8_t* d_bytes, const uint64_t* h_byte_off,
                   const uint64_t* h_nbits, int16_t* d_coef, void* stream);

/* Restart records -- an EXTENSION beside the reference's format, which carries none (codec.py:319-334;
 * hiccup_b200/hicimage.py appends them to a `.hic` file as one extra list entry the reference's reader never
 * looks at).  For every 128-bit subsequence of every bit stream, in stream order: `off` = how many bits past the
 * subsequence's upper boundary the next codeword starts, `cnt` = how many codewords start inside its span.
 *   hic_decode_sync             runs only the synchronisation passes of D1 over the streams (n_sub_out =
 *                               subsequences in all streams: 128-bit pieces of 8 + nbits bits each);
 *   hic_decode_export_restarts  the records the most recent run or sync converged to, into host arrays;
 *   hic_decode_run_restarts     hic_decode_run without the synchronisation passes.  Every span is still
 *                               checked against its record: records that do not fit the streams give
 *                               HIC_ERR_CORRUPT, never a silent mis-decode. */
int hic_decode_sync(hic_decode_plan* plan, const uint8_t* d_bytes, const uint64_t* h_byte_off, const uint64_t* h_nbits,
                    uint64_t* n_sub_out, void* stream);
int hic_decode_export_restarts(hic_decode_plan* plan, uint8_t* h_off, uint8_t* h_cnt, uint64_t capacity, void* stream);
int hic_decode_run_restarts(hic_decode_plan* plan, const uint8_t* d_bytes, const uint64_t* h_byte_off,
                            const uint64_t* h_nbits, const uint8_t* h_off, const uint8_t* h_cnt, uint64_t n_sub,
                            int16_t* d_coef, void* stream);

/* DC-only decode (DCT layouts; a flat layout gives HIC_ERR_INVALID) -- the DC half of codec.jpeg_decode
 * (codec.py:337-426): HuffmanTree.decode_data (huffman.py:149-174) of the three DC bit strings of every image
 * and utils.invert_differences (utils.py:66-74).  Only the kind-0 streams are read: the offsets, bit counts
 * and bytes of kinds 1 and 2 are ignored (their tables may have no rows), and hic_decode_set_data_bytes
 * bounds apply to the DC streams.  d_dc receives one int16 DC value per block, index image *
 * blocks_per_image + block.  h_off / h_cnt / n_sub: the restart records of the DC streams alone, in stream
 * order, or NULL / NULL / 0 to synchronise.  Synchronises `stream`; HIC_ERR_CORRUPT if a DC stream does
 * not decode to exactly one symbol per block of its channel (or the records do not belong to it). */
int hic_decode_run_dc(hic_decode_plan* plan, const uint8_t* d_bytes, const uint64_t* h_byte_off, const uint64_t* h_nbits,
                      const uint8_t* h_off, const uint8_t* h_cnt, uint64_t n_sub, int16_t* d_dc, void* stream);

/* ---- host-side helpers of the `.hic` container (no device involved) -------------------------------------
 * The rows of one Huffman table to / from the byte strings the reference pickles them as, one pickle per row
 * (hicimage.py:57-60, 103-121: TupP.byte_stream inside PayloadStringP).  numpy_scalar[i] != 0 (NULL: none): row i's symbol
 * is a numpy.int32 scalar (DC tables, non-zero wavelet values), written as <np_pre> <4 value bytes> <np_mid> -- the bytes this environment's numpy puts
 * around them, which hiccup_b200/hicimage.py reads off a sample pickle.  pack: row i is out[out_off[i] ..
 * out_off[i + 1]) (out_off has n + 1 entries).  parse: accepts exactly the canonical forms; *bad_row = the first
 * row that is anything else (the caller then unpickles the table the slow way), -1 if none. */
int hic_hicfile_pack_rows(const int32_t* symbols, const uint8_t* lens, const uint64_t* codes, uint64_t n, const uint8_t* numpy_scalar,
                          const uint8_t* np_pre, uint32_t np_pre_len, const uint8_t* np_mid, uint32_t np_mid_len,
                          uint8_t* out, uint64_t out_capacity, uint64_t* out_off);
int hic_hicfile_parse_rows(const uint8_t* data, const uint64_t* off, uint64_t n, const uint8_t* np_pre, uint32_t np_pre_len,
                           const uint8_t* np_mid, uint32_t np_mid_len, int32_t* symbols, uint8_t* lens, uint64_t* codes,
                           uint8_t* numpy_scalar, int64_t* bad_row);
/* A whole table payload, byte-identical to pickle.dumps({"type": TupP, "data": [row pickles]}) (hicimage.py:103-121:
 * PayloadStringP.byte_stream) under protocol 4: `head` = the pickle's bytes from the dict's opcode up to the list's MEMOIZE
 * (they name the TupP class; read off a sample pickle by hiccup_b200/hicimage.py), then the rows as memoised bytes
 * objects in batches of 1000, in 64 KiB frames as CPython's pickler cuts them.  *out_len = the payload's size. */
int hic_hicfile_pack_table(const int32_t* symbols, const uint8_t* lens, const uint64_t* codes, uint64_t n, const uint8_t* numpy_scalar,
                           const uint8_t* np_pre, uint32_t np_pre_len, const uint8_t* np_mid, uint32_t np_mid_len,
                           const uint8_t* head, uint32_t head_len, uint8_t* out, uint64_t out_capacity, uint64_t* out_len);
/* The reverse (hicimage.py:97-101: PayloadStringP.from_bytes): walks a table payload written by pickle protocol 4 or 5 whose
 * "type" is <any package>.hicimage.TupP and fills the row arrays (row_capacity entries each; size / 23 rows always
 * suffice).  *canonical = 1 and *n_rows = the row count when every opcode and row is of the canonical form, else
 * *canonical = 0 (the caller then unpickles the payload the slow way; nothing is trusted from the arrays). */
int hic_hicfile_parse_table(const uint8_t* data, uint64_t size, const uint8_t* np_pre, uint32_t np_pre_len, const uint8_t* np_mid,
                            uint32_t np_mid_len, int32_t* symbols, uint8_t* lens, uint64_t* codes, uint8_t* numpy_scalar,
                            uint64_t row_capacity, uint64_t* n_rows, int32_t* canonical);

/* Whole `.hic` files of a batch, written by host threads (hicimage.py:165-183: pickle.dump(HicImage.byte_stream(), f), i.e.
 * the pickled list [type string, table payloads, framed bit strings, shapes]).  env: what this environment's pickle and
 * numpy write around the data (read off sample pickles by hiccup_b200/hicimage.py, which also checks these functions
 * against pickle.dumps before using them).  batch: file i's k-th table and k-th bit string are symbol stream
 * stream_of[i * tables_per_file + k] of an encode result in the layout of hic_entropy_tables_packed + the framed payloads
 * of hic_entropy_pack; flag_mode[k]: 0 the table's symbols are Python ints, 1 numpy.int32 scalars (DC tables), 2
 * numpy.int32 unless the symbol is 0 (wavelet value tables); lead: the first list entry (the mode string); trail: the
 * n_trail entries after the bit strings (the two shape pickles), concatenated.
 * files_bound: bound[i] = room that always suffices for file i.  pack_files: file i goes to out[out_off[i] ..) (room
 * out_off[i + 1] - out_off[i]), its size to out_len[i]; out_len[i] = 0: left to the caller (an entry shorter than two
 * bytes, which pickle may write as a memo reference).  threads: host threads to use (files are independent). */
typedef struct hic_hicfile_env {
    const uint8_t* np_pre;
    const uint8_t* np_mid;
    const uint8_t* head;
    uint32_t np_pre_len, np_mid_len, head_len, reserved;
} hic_hicfile_env;
typedef struct hic_hicfile_batch {
    uint64_t n_files;
    uint32_t tables_per_file, n_trail;
    const uint32_t* stream_of;
    const uint8_t* flag_mode;
    const uint32_t* index;
    const int32_t* symbols;
    const uint64_t* packed;
    const uint8_t* data;
    const uint64_t* byte_off;
    const uint64_t* byte_len;
    const uint8_t* lead;
    uint64_t lead_len;
    const uint8_t* trail;
    const uint64_t* trail_len;
} hic_hicfile_batch;
int hic_hicfile_files_bound(const hic_hicfile_env* env, const hic_hicfile_batch* batch, uint64_t* bound, uint32_t threads);
int hic_hicfile_pack_files(const hic_hicfile_env* env, const hic_hicfile_batch* batch, uint8_t* out, const uint64_t* out_off,
                           uint64_t* out_len, uint32_t threads);
/* The reverse, for a batch of files in host memory (file i = file_len[i] bytes at files[i]), in two steps so that
 * the caller can size the arrays exactly.  scan: positions (from the file's start) and sizes of each file's first n_items
 * entries -- entry 0 the mode string, 1 .. T the tables, T + 1 .. 2T the bit strings, then the shapes -- and the row count
 * of every table; canonical[i] = 0 where file i is not the plain list of byte strings pickle protocol 4 / 5 writes (the
 * caller reads such files with the unpickler).  parse: table k of file i goes to rows index[2 s] .. + index[2 s + 1] of
 * symbols / packed (the layout hic_decode_set_tables_packed takes; s = stream_of[i * T + k]; the counts must be scan's),
 * its bit string to data + byte_off[s] and its payload bit count (iohelper.py: the signed pad byte) to nbits[s];
 * ok[i] = 0 if a row of file i is not of the canonical form. */
int hic_hicfile_scan_files(const uint8_t* const* files, const uint64_t* file_len, uint64_t n_files, uint32_t tables_per_file, uint32_t n_items,
                           uint64_t* item_off, uint64_t* item_len, uint32_t* rows, uint8_t* canonical, uint32_t threads);
int hic_hicfile_parse_files(const hic_hicfile_env* env, const uint8_t* const* files, uint64_t n_files, uint32_t tables_per_file, uint32_t n_items,
                            const uint64_t* item_off, const uint64_t* item_len, const uint32_t* stream_of, const uint32_t* index,
                            int32_t* symbols, uint64_t* packed, uint8_t* data, const uint64_t* byte_off, uint64_t* nbits,
                            uint8_t* ok, uint32_t threads);

#ifdef __cplusplus
}
#endif
#endif /* HICCUP_B200_H */
