// hic_wavelet_general.cu -- wavelet ("HIC") mode at settings other than the defaults: any
// WAVELET_NUM_LEVELS in 1..5, any WAVELET_SUBBAND_QUANTIZATION_MULTIPLIER != 0, any WAVELET_THRESHOLD,
// WAVELET_QUALITY_FACTOR < 1 (reference settings.py:12-16), for the db1 / haar filter pair
// (model.py:31-35; "haar" is PyWavelets' alias of "db1").  hic_wavelet.cu is the fused fast path for the
// default settings; this file is the level-by-level general path with the same arithmetic.
//
// Reference: compression.wavelet_compression (compression.py:59-85), quantization.subband_quantize /
// subband_invert_quantize (quantization.py:60-77), transform.threshold_channel_by_quality +
// quantization.quality_threshold_value (transform.py:242-250, quantization.py:84-94: an order statistic
// over ALL coefficients of a channel), transform.threshold (transform.py:227-239),
// compression.wavelet_decompression (compression.py:88-100).  The transform is PyWavelets' wavedec2 /
// waverec2 restated in float64 (oracle/pywt_standin.py) -- PARITY UNPINNED against the real package.
//
// Forward, per image and channel:  colour -> (x - 256) as float64 plane; for l = 1..L one kernel turns the
// (h_{l-1} x w_{l-1}) approximation plane into the (h_l x w_l) one and writes the three detail bands,
// divided by multiplier * (i*i + 1) (i = L - l) and rounded half-even, at their zigzag positions of the
// flat stream; cA_L is rounded.  With a quality factor below 1 the thresholds wait: a 65536-bin histogram
// of the channel's quantised coefficients gives the order statistic s[thresh_index] (a radix select with
// one 16-bit digit: the flat stream is int16), then one pass zeroes |v| < that value and |v| < threshold.
// HBM-bound integer / float64 streaming work, one thread per output sample; not the benchmarked path.
#include "hic_core.cuh"
#include "hic_runtime.cuh"
#include "hic_wavelet_common.cuh"

namespace hic {
namespace wvg {

constexpr double C = 0x1.6a09e667f3bcdp-1;   // PyWavelets' db1 coefficient as a double
constexpr int HIST_BINS = 65536;

struct Pyr {
    hic_wavelet_pyramid p;
    int64_t chan_elems;          // 64 * ceil(len / 64)
};

static int pyramid_of(int h, int w, int levels, hic_wavelet_pyramid* g) {
    HIC_REQUIRE(g != nullptr, "pyramid output is NULL");
    HIC_REQUIRE(h >= 1 && w >= 1 && h <= 65536 && w <= 65536, "image must be 1..65536 on a side (got %dx%d)", h, w);
    HIC_REQUIRE(levels >= 1 && levels <= HIC_WAVELET_MAX_LEVELS, "WAVELET_NUM_LEVELS must be in 1..%d (got %d)",
                HIC_WAVELET_MAX_LEVELS, levels);
    g->h = h;
    g->w = w;
    g->levels = levels;
    g->n_bands = 3 * levels + 1;
    g->lh[0] = h;
    g->lw[0] = w;
    for (int l = 1; l <= HIC_WAVELET_MAX_LEVELS; ++l) {     // pywt.dwt_coeff_len for db1, symmetric mode: ceil(n / 2)
        g->lh[l] = l <= levels ? (g->lh[l - 1] + 1) / 2 : 0;
        g->lw[l] = l <= levels ? (g->lw[l - 1] + 1) / 2 : 0;
    }
    int64_t off = 0;
    for (int b = 0; b < 16; ++b) {
        g->band_off[b] = off;
        if (b < g->n_bands) {
            const int lvl = b == 0 ? levels : levels - (b - 1) / 3;
            off += (int64_t)g->lh[lvl] * g->lw[lvl];
        }
    }
    g->len = off;
    return HIC_OK;
}

__host__ __device__ inline int band_level(int band, int levels) { return band == 0 ? levels : levels - (band - 1) / 3; }

static int make(int h, int w, int levels, Pyr* g) {
    const int rc = pyramid_of(h, w, levels, &g->p);
    if (rc) return rc;
    g->chan_elems = 64 * ((g->p.len + 63) / 64);
    return HIC_OK;
}

static inline unsigned blocks_for(int64_t items) { return (unsigned)((items + 255) / 256); }

// ---- forward ----
__global__ void __launch_bounds__(256)
colour_kernel(const uint8_t* __restrict__ rgb, int64_t pixels, int64_t total, double* __restrict__ plane) {
    const int64_t gid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= total) return;
    const int64_t img = gid / pixels, p = gid - img * pixels;
    const uint8_t* s = rgb + gid * 3;
    int y, cr, cb;
    rgb_to_ycrcb(s[0], s[1], s[2], y, cr, cb);
    double* o = plane + img * 3 * pixels + p;
    o[0] = (double)(y - 256);                 // compression.py:70: x - 2^8
    o[pixels] = (double)(cr - 256);
    o[2 * pixels] = (double)(cb - 256);
}

__device__ __forceinline__ void haar_pair(double even, double odd, double& a, double& d) {
    const double ce = dmul(C, even), co = dmul(C, odd);
    a = dadd(co, ce);              // (c * x[2k+1]) + (c * x[2k])
    d = dadd(-co, ce);             // (-c * x[2k+1]) + (c * x[2k])
}

__device__ __forceinline__ int16_t quantise(double v, double div, double thr) {
    const int q = __double2int_rn(ddiv(v, div));          // np.divide, np.round (half even), astype(int32)
    return (int16_t)((fabs((double)q) < thr) ? 0 : q);
}

// one decomposition level: in (hi x wi) -> aa (ho x wo) + three quantised detail bands
__global__ void __launch_bounds__(256)
level_kernel(const double* __restrict__ in, int hi, int wi, int64_t in_stride, double* __restrict__ aa, int ho, int wo,
             int64_t out_stride, int64_t n3, Pyr g, int band0, double div, double thr, int16_t* __restrict__ flat) {
    const int64_t per = (int64_t)ho * wo;
    const int64_t gid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= per * n3) return;
    const int64_t cs = gid / per;
    const int64_t e = gid - cs * per;
    const int k = (int)(e / wo), j = (int)(e - (int64_t)k * wo);
    const double* src = in + cs * in_stride;
    const int r0 = 2 * k, r1 = min(2 * k + 1, hi - 1);          // symmetric extension: x[N] = x[N-1]
    const int c0 = 2 * j, c1 = min(2 * j + 1, wi - 1);
    double a_l, d_l, a_r, d_r;                                   // axis 0 first (pywt.dwtn)
    haar_pair(src[(int64_t)r0 * wi + c0], src[(int64_t)r1 * wi + c0], a_l, d_l);
    haar_pair(src[(int64_t)r0 * wi + c1], src[(int64_t)r1 * wi + c1], a_r, d_r);
    double v_aa, v_ad, v_da, v_dd;
    haar_pair(a_l, a_r, v_aa, v_ad);
    haar_pair(d_l, d_r, v_da, v_dd);
    aa[cs * out_stride + e] = v_aa;
    int16_t* dst = flat + cs * g.chan_elems;
    const int64_t pos = zigzag_pos(k, j, ho, wo);
    dst[g.p.band_off[band0] + pos] = quantise(v_da, div, thr);           // cH = 'da'
    dst[g.p.band_off[band0 + 1] + pos] = quantise(v_ad, div, thr);       // cV = 'ad'
    dst[g.p.band_off[band0 + 2] + pos] = quantise(v_dd, div, thr);       // cD = 'dd'
}

__global__ void __launch_bounds__(256)
approximation_kernel(const double* __restrict__ aa, int ho, int wo, int64_t stride, int64_t n3, Pyr g, double thr,
                     int16_t* __restrict__ flat) {
    const int64_t per = (int64_t)ho * wo;
    const int64_t gid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= per * n3) return;
    const int64_t cs = gid / per;
    const int64_t e = gid - cs * per;
    const int k = (int)(e / wo), j = (int)(e - (int64_t)k * wo);
    flat[cs * g.chan_elems + zigzag_pos(k, j, ho, wo)] = quantise(aa[cs * stride + e], 1.0, thr);
}

__global__ void __launch_bounds__(256)
histogram_kernel(const int16_t* __restrict__ flat, Pyr g, int64_t n3, uint32_t* __restrict__ hist) {
    const int64_t gid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= g.p.len * n3) return;
    const int64_t cs = gid / g.p.len;
    const int64_t e = gid - cs * g.p.len;
    atomicAdd(&hist[cs * HIST_BINS + ((int)flat[cs * g.chan_elems + e] + 32768)], 1u);
}

// s[thresh_index] of the ascending signed sort of a channel's coefficients (quantization.py:90-94)
__global__ void __launch_bounds__(1024)
select_kernel(const uint32_t* __restrict__ hist, int64_t thresh_index, int32_t* __restrict__ value) {
    __shared__ unsigned long long part[1024];
    const uint32_t* hs = hist + (int64_t)blockIdx.x * HIST_BINS;
    constexpr int PER = HIST_BINS / 1024;
    unsigned long long mine = 0;
    for (int b = 0; b < PER; ++b) mine += hs[threadIdx.x * PER + b];
    part[threadIdx.x] = mine;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long before = 0;
        int t = 0;
        while (t < 1023 && before + part[t] <= (unsigned long long)thresh_index) before += part[t++];
        int b = t * PER;
        while (b < HIST_BINS - 1 && before + hs[b] <= (unsigned long long)thresh_index) before += hs[b++];
        value[blockIdx.x] = b - 32768;
    }
}

__global__ void __launch_bounds__(256)
threshold_kernel(int16_t* __restrict__ flat, Pyr g, int64_t n3, const int32_t* __restrict__ value, double thr) {
    const int64_t gid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= g.p.len * n3) return;
    const int64_t cs = gid / g.p.len;
    const int64_t e = gid - cs * g.p.len;
    int16_t* p = flat + cs * g.chan_elems + e;
    const int v = *p, a = v < 0 ? -v : v;
    if (a < value[cs] || (double)a < thr) *p = 0;           // transform.py:227-239, twice (compression.py:76-79)
}

// ---- inverse ----
__global__ void __launch_bounds__(256)
approximation_load_kernel(const int16_t* __restrict__ flat, Pyr g, int ho, int wo, int64_t stride, int64_t n3,
                          double* __restrict__ aa) {
    const int64_t per = (int64_t)ho * wo;
    const int64_t gid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= per * n3) return;
    const int64_t cs = gid / per;
    const int64_t e = gid - cs * per;
    const int k = (int)(e / wo), j = (int)(e - (int64_t)k * wo);
    aa[cs * stride + e] = (double)flat[cs * g.chan_elems + zigzag_pos(k, j, ho, wo)];
}

__device__ __forceinline__ void ihaar_pair(double a, double d, double& even, double& odd) {
    const double ca = dmul(C, a), cd = dmul(C, d);
    even = dadd(ca, cd);
    odd = dadd(ca, -cd);
}

// one reconstruction step at the position whose zigzag index in the level's bands is `pos`: the approximation
// sample v_aa and the three detail coefficients there, times `mul` (quantization.py:72-77) -> the 2 x 2 children
// q[row][col] of the next finer level
__device__ __forceinline__ void inverse_quad(double v_aa, const int16_t* __restrict__ src, const Pyr& g, int band0, int64_t pos,
                                             double mul, double (&q)[2][2]) {
    const double v_da = dmul((double)src[g.p.band_off[band0] + pos], mul);
    const double v_ad = dmul((double)src[g.p.band_off[band0 + 1] + pos], mul);
    const double v_dd = dmul((double)src[g.p.band_off[band0 + 2] + pos], mul);
    double a_e, a_o, d_e, d_o;                                                    // idwtn undoes the LAST axis first
    ihaar_pair(v_aa, v_ad, a_e, a_o);
    ihaar_pair(v_da, v_dd, d_e, d_o);
    ihaar_pair(a_e, d_e, q[0][0], q[1][0]);
    ihaar_pair(a_o, d_o, q[0][1], q[1][1]);
}

// one reconstruction level: aa (ho x wo) + the level's detail bands times `mul` -> out (H x W), H = 2 ho or
// 2 ho - 1: pywt.waverec2 trims the extra row / column when the next detail band is one smaller
__global__ void __launch_bounds__(256)
inverse_level_kernel(const double* __restrict__ aa, int ho, int wo, int64_t in_stride, double* __restrict__ out, int H, int W,
                     int64_t n3, Pyr g, int band0, double mul, const int16_t* __restrict__ flat) {
    const int64_t per = (int64_t)ho * wo;
    const int64_t gid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= per * n3) return;
    const int64_t cs = gid / per;
    const int64_t e = gid - cs * per;
    const int k = (int)(e / wo), j = (int)(e - (int64_t)k * wo);
    const int16_t* src = flat + cs * g.chan_elems;
    const int64_t pos = zigzag_pos(k, j, ho, wo);
    const double v_aa = aa[cs * in_stride + e];
    double q[2][2];
    inverse_quad(v_aa, src, g, band0, pos, mul, q);
    double* o = out + cs * ((int64_t)H * W);
    const bool row1 = 2 * k + 1 < H, col1 = 2 * j + 1 < W;
    o[(int64_t)(2 * k) * W + 2 * j] = q[0][0];
    if (row1) o[(int64_t)(2 * k + 1) * W + 2 * j] = q[1][0];
    if (col1) o[(int64_t)(2 * k) * W + 2 * j + 1] = q[0][1];
    if (row1 && col1) o[(int64_t)(2 * k + 1) * W + 2 * j + 1] = q[1][1];
}

// one channel sample: + 2^8, astype(uint8): truncate, wrap (compression.py:95)
__device__ __forceinline__ int finish_sample(double v) { return wrap_u8(dadd(v, 256.0)); }

__device__ __forceinline__ void store_pixel(int y, int cr, int cb, uint8_t* __restrict__ o) {
    int r, gg, b;
    ycrcb_to_rgb(y, cr, cb, r, gg, b);
    o[0] = (uint8_t)r;
    o[1] = (uint8_t)gg;
    o[2] = (uint8_t)b;
}

__global__ void __launch_bounds__(256)
finish_kernel(const double* __restrict__ plane, int64_t pixels, int64_t total, uint8_t* __restrict__ rgb) {
    const int64_t gid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= total) return;
    const int64_t img = gid / pixels, p = gid - img * pixels;
    const double* s = plane + img * 3 * pixels + p;
    store_pixel(finish_sample(s[0]), finish_sample(s[pixels]), finish_sample(s[2 * pixels]), rgb + gid * 3);
}

// finish_kernel for the 1/s-scale image: the running approximation A_k (s = 2^k) times 2^-k (exact) is the mean of
// each s x s tile of the unrounded image
__global__ void __launch_bounds__(256)
scaled_finish_kernel(const double* __restrict__ plane, int64_t pixels, int64_t total, double inv_scale, uint8_t* __restrict__ rgb) {
    const int64_t gid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= total) return;
    const int64_t img = gid / pixels, p = gid - img * pixels;
    const double* s = plane + img * 3 * pixels + p;
    store_pixel(finish_sample(dmul(s[0], inv_scale)), finish_sample(dmul(s[pixels], inv_scale)),
                finish_sample(dmul(s[2 * pixels], inv_scale)), rgb + gid * 3);
}

// ---- region: one rh x rw window of the 1/s-scale image (s = 2^k, 0 <= k <= L) per image ----
// db1 has no halo: a level-(l-1) sample at (y, x) reads only the level-l approximation at (y >> 1, x >> 1) and the
// three detail coefficients there.  So a window needs, at each level l > k, only the dyadic parent rectangle of its
// rows [top >> (l-k), (top+rh-1) >> (l-k)] (columns alike), and every sample on that path is the very float64 value
// the full inverse computes at that position.
struct RegionArgs {
    const int32_t* origin;         // (top, left) per image, in the coordinates of the 1/s image
    int n, rh, rw;
    double mul[HIC_WAVELET_MAX_LEVELS];   // detail group i's dequantisation factor (0 = coarsest)
    double inv_scale;              // 2^-k
};

// D = L - k levels to reconstruct.  D = 0: one thread per window pixel, straight from cA_L.  D >= 1: one thread per
// level-(k+1) sample of the window's parent rectangle (a 2 x 2 output quad), all three channels (ycrcb_to_rgb needs
// them together); per channel it starts from cA_L, keeps only the child on its own path through levels L .. k+2, and
// finishes with inverse_level_kernel's quad.  No float64 planes, no intermediate traffic.
template <int D>
__global__ void __launch_bounds__(256)
region_kernel(const int16_t* __restrict__ flat, Pyr g, RegionArgs a, uint8_t* __restrict__ rgb) {
    constexpr int Q = D == 0 ? 1 : 2;                  // output pixels per thread along each axis
    const int L = g.p.levels, k = L - D;
    const int ph = D == 0 ? a.rh : a.rh / 2 + 1, pw = D == 0 ? a.rw : a.rw / 2 + 1;
    const int64_t per = (int64_t)ph * pw;
    const int64_t gid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= per * a.n) return;
    const int64_t img = gid / per;
    const int rem = (int)(gid - img * per);
    const int top = __ldg(a.origin + 2 * img), left = __ldg(a.origin + 2 * img + 1);
    // this thread's position at level k + (D > 0): the window pixel itself, or the parent of a quad
    const int py = (D == 0 ? top : top >> 1) + rem / pw, px = (D == 0 ? left : left >> 1) + rem % pw;
    if (Q * py > top + a.rh - 1 || Q * px > left + a.rw - 1) return;
    int u[3][Q][Q];                                   // finished samples, by channel
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        const int16_t* src = flat + (3 * img + c) * g.chan_elems;
        double s = (double)src[g.p.band_off[0] + zigzag_pos(py >> (D > 0 ? D - 1 : 0), px >> (D > 0 ? D - 1 : 0), g.p.lh[L], g.p.lw[L])];
        if constexpr (D == 0) {
            u[c][0][0] = finish_sample(dmul(s, a.inv_scale));
        } else {
            double q[2][2];
#pragma unroll
            for (int i = 0; i < D - 1; ++i) {          // level L - i -> L - i - 1, keeping the child on this path
                const int sh = D - 1 - i, l = L - i;
                inverse_quad(s, src, g, 1 + 3 * i, zigzag_pos(py >> sh, px >> sh, g.p.lh[l], g.p.lw[l]), a.mul[i], q);
                const bool ry = (py >> (sh - 1)) & 1, rx = (px >> (sh - 1)) & 1;     // selects, not a local-memory index
                s = ry ? (rx ? q[1][1] : q[1][0]) : (rx ? q[0][1] : q[0][0]);
            }
            inverse_quad(s, src, g, 1 + 3 * (D - 1), zigzag_pos(py, px, g.p.lh[k + 1], g.p.lw[k + 1]), a.mul[D - 1], q);
#pragma unroll
            for (int dy = 0; dy < 2; ++dy)
#pragma unroll
                for (int dx = 0; dx < 2; ++dx) u[c][dy][dx] = finish_sample(dmul(q[dy][dx], a.inv_scale));
        }
    }
    uint8_t* dst = rgb + (size_t)img * a.rh * a.rw * 3;
#pragma unroll
    for (int dy = 0; dy < Q; ++dy)
#pragma unroll
        for (int dx = 0; dx < Q; ++dx) {
            const int oy = Q * py + dy, ox = Q * px + dx;
            if (oy < top || oy >= top + a.rh || ox < left || ox >= left + a.rw) continue;
            store_pixel(u[0][dy][dx], u[1][dy][dx], u[2][dy][dx], dst + ((size_t)(oy - top) * a.rw + (ox - left)) * 3);
        }
}

// ---- layout converters: flat zigzag stream <-> 3 L + 1 raster int32 sub-bands ----
__global__ void __launch_bounds__(256)
flat_to_bands_kernel(const int16_t* __restrict__ flat, Pyr g, int64_t n3, int32_t* __restrict__ bands) {
    const int64_t per = g.p.len;
    const int64_t gid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= per * n3) return;
    const int64_t cs = gid / per;
    const int64_t e = gid - cs * per;
    int band = g.p.n_bands - 1;
    while (e < g.p.band_off[band]) --band;
    const int lvl = band_level(band, g.p.levels);
    const int hb = g.p.lh[lvl], wb = g.p.lw[lvl];
    const int64_t r = e - g.p.band_off[band];
    const int y = (int)(r / wb), x = (int)(r - (int64_t)y * wb);
    bands[gid] = (int32_t)flat[cs * g.chan_elems + g.p.band_off[band] + zigzag_pos(y, x, hb, wb)];
}

__global__ void __launch_bounds__(256)
bands_to_flat_kernel(const int32_t* __restrict__ bands, Pyr g, int64_t n3, int16_t* __restrict__ flat) {
    const int64_t per = g.p.len;
    const int64_t gid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= per * n3) return;
    const int64_t cs = gid / per;
    const int64_t e = gid - cs * per;
    int band = g.p.n_bands - 1;
    while (e < g.p.band_off[band]) --band;
    const int lvl = band_level(band, g.p.levels);
    const int hb = g.p.lh[lvl], wb = g.p.lw[lvl];
    const int64_t r = e - g.p.band_off[band];
    const int y = (int)(r / wb), x = (int)(r - (int64_t)y * wb);
    flat[cs * g.chan_elems + g.p.band_off[band] + zigzag_pos(y, x, hb, wb)] = (int16_t)bands[gid];
}

static int check_params(const hic_wavelet_params* p) {
    HIC_REQUIRE(p != nullptr, "params is NULL");
    HIC_REQUIRE(p->levels >= 1 && p->levels <= HIC_WAVELET_MAX_LEVELS, "WAVELET_NUM_LEVELS must be in 1..%d (got %d)",
                HIC_WAVELET_MAX_LEVELS, p->levels);
    HIC_REQUIRE(p->multiplier != 0.0 && p->multiplier == p->multiplier, "WAVELET_SUBBAND_QUANTIZATION_MULTIPLIER must be a non-zero number");
    HIC_REQUIRE(p->threshold >= 0.0, "WAVELET_THRESHOLD must be >= 0");
    return HIC_OK;
}

static size_t plane_doubles(int n, int h, int w) { return (size_t)n * 3 * h * w; }

}  // namespace wvg
}  // namespace hic

extern "C" {

int hic_wavelet_pyramid_of(int32_t h, int32_t w, int32_t levels, hic_wavelet_pyramid* out) {
    return hic::wvg::pyramid_of(h, w, levels, out);
}

int hic_wavelet_general_work_bytes(int32_t n, int32_t h, int32_t w, size_t* out) {
    using namespace hic;
    HIC_REQUIRE(out != nullptr, "output is NULL");
    HIC_REQUIRE(n >= 1 && h >= 1 && w >= 1, "bad shape");
    // two float64 plane sets (ping-pong between levels) + the per-channel histograms and selected values
    *out = 2 * wvg::plane_doubles(n, h, w) * sizeof(double) + (size_t)n * 3 * (wvg::HIST_BINS + 16) * sizeof(uint32_t);
    return HIC_OK;
}

int hic_wavelet_forward_general(const uint8_t* d_rgb, int32_t n, int32_t h, int32_t w, const hic_wavelet_params* params,
                                void* d_work, int16_t* d_flat, void* stream) {
    using namespace hic;
    HIC_REQUIRE(d_rgb && d_flat && d_work, "NULL device pointer");
    HIC_REQUIRE(n >= 1 && n <= 65535, "batch size must be in 1..65535 (got %d)", n);
    int rc = wvg::check_params(params);
    if (rc) return rc;
    wvg::Pyr g;
    rc = wvg::make(h, w, params->levels, &g);
    if (rc) return rc;
    const int L = params->levels;
    HIC_REQUIRE(params->threshold_index < g.p.len, "threshold index %lld is past the %lld coefficients of a channel",
                (long long)params->threshold_index, (long long)g.p.len);
    cudaStream_t st = as_stream(stream);
    const int64_t n3 = 3 * (int64_t)n, pixels = (int64_t)h * w;
    double* plane[2] = {static_cast<double*>(d_work), static_cast<double*>(d_work) + wvg::plane_doubles(n, h, w)};
    uint32_t* hist = reinterpret_cast<uint32_t*>(plane[1] + wvg::plane_doubles(n, h, w));
    int32_t* value = reinterpret_cast<int32_t*>(hist + (size_t)n3 * wvg::HIST_BINS);
    const bool select = params->threshold_index >= 0;               // WAVELET_QUALITY_FACTOR < 1
    const double thr = select ? 0.0 : params->threshold;            // (the thresholds wait for the order statistic)
    HIC_CUDA(cudaMemsetAsync(d_flat, 0, (size_t)g.chan_elems * n3 * sizeof(int16_t), st));
    HIC_LAUNCH("wavelet_colour_kernel", st, wvg::colour_kernel<<<wvg::blocks_for(pixels * n), 256, 0, st>>>(d_rgb, pixels, pixels * n, plane[0]));
    int cur = 0;
    for (int l = 1; l <= L; ++l) {
        const int hi = g.p.lh[l - 1], wi = g.p.lw[l - 1], ho = g.p.lh[l], wo = g.p.lw[l];
        const int i = L - l;                                        // quantization.py:65-68: hfs[i], i = 0 the coarsest
        const double div = params->multiplier * (double)(i * i + 1);
        HIC_LAUNCH("wavelet_level_kernel", st, wvg::level_kernel<<<wvg::blocks_for((int64_t)ho * wo * n3), 256, 0, st>>>(
            plane[cur], hi, wi, (int64_t)hi * wi, plane[cur ^ 1], ho, wo, (int64_t)ho * wo, n3, g, 1 + 3 * i, div, thr, d_flat));
        cur ^= 1;
    }
    HIC_LAUNCH("wavelet_approximation_kernel", st, wvg::approximation_kernel<<<wvg::blocks_for((int64_t)g.p.lh[L] * g.p.lw[L] * n3), 256, 0, st>>>(
        plane[cur], g.p.lh[L], g.p.lw[L], (int64_t)g.p.lh[L] * g.p.lw[L], n3, g, thr, d_flat));
    if (select) {
        HIC_CUDA(cudaMemsetAsync(hist, 0, (size_t)n3 * wvg::HIST_BINS * sizeof(uint32_t), st));
        HIC_LAUNCH("wavelet_histogram_kernel", st, wvg::histogram_kernel<<<wvg::blocks_for(g.p.len * n3), 256, 0, st>>>(d_flat, g, n3, hist));
        HIC_LAUNCH("wavelet_select_kernel", st, wvg::select_kernel<<<(unsigned)n3, 1024, 0, st>>>(hist, params->threshold_index, value));
        HIC_LAUNCH("wavelet_threshold_kernel", st, wvg::threshold_kernel<<<wvg::blocks_for(g.p.len * n3), 256, 0, st>>>(d_flat, g, n3, value, params->threshold));
    }
    return HIC_OK;
}

int hic_wavelet_inverse_general(const int16_t* d_flat, int32_t n, int32_t h, int32_t w, const hic_wavelet_params* params,
                                void* d_work, uint8_t* d_rgb_out, void* stream) {
    using namespace hic;
    HIC_REQUIRE(d_rgb_out && d_flat && d_work, "NULL device pointer");
    HIC_REQUIRE(n >= 1 && n <= 65535, "batch size must be in 1..65535 (got %d)", n);
    int rc = wvg::check_params(params);
    if (rc) return rc;
    const int L = params->levels;
    HIC_REQUIRE(h % 2 == 0 && w % 2 == 0, "the reconstructed image is 2 ceil(h / 2) x 2 ceil(w / 2): pass even sides (got %dx%d)", h, w);
    wvg::Pyr g;
    rc = wvg::make(h, w, L, &g);
    if (rc) return rc;
    cudaStream_t st = as_stream(stream);
    const int64_t n3 = 3 * (int64_t)n, pixels = (int64_t)h * w;
    double* plane[2] = {static_cast<double*>(d_work), static_cast<double*>(d_work) + wvg::plane_doubles(n, h, w)};
    int cur = L & 1;                                                // so that the last level lands in plane[0]
    HIC_LAUNCH("wavelet_approximation_load_kernel", st, wvg::approximation_load_kernel<<<wvg::blocks_for((int64_t)g.p.lh[L] * g.p.lw[L] * n3), 256, 0, st>>>(
        d_flat, g, g.p.lh[L], g.p.lw[L], (int64_t)g.p.lh[L] * g.p.lw[L], n3, plane[cur]));
    for (int l = L; l >= 1; --l) {
        const int ho = g.p.lh[l], wo = g.p.lw[l];
        const int i = L - l;
        const double mul = params->multiplier * (double)(i * i + 1);
        HIC_LAUNCH("wavelet_inverse_level_kernel", st, wvg::inverse_level_kernel<<<wvg::blocks_for((int64_t)ho * wo * n3), 256, 0, st>>>(
            plane[cur], ho, wo, (int64_t)ho * wo, plane[cur ^ 1], g.p.lh[l - 1], g.p.lw[l - 1], n3, g, 1 + 3 * i, mul, d_flat));
        cur ^= 1;
    }
    // plane[cur] holds channel-planar float64 samples; its (image, channel) stride is h * w
    HIC_LAUNCH("wavelet_finish_kernel", st, wvg::finish_kernel<<<wvg::blocks_for(pixels * n), 256, 0, st>>>(plane[cur], pixels, pixels * n, d_rgb_out));
    return HIC_OK;
}

int hic_wavelet_scaled_general(const int16_t* d_flat, int32_t n, int32_t h, int32_t w, const hic_wavelet_params* params,
                               int32_t scale, void* d_work, uint8_t* d_rgb_out, void* stream) {
    using namespace hic;
    HIC_REQUIRE(d_rgb_out && d_flat && d_work, "NULL device pointer");
    HIC_REQUIRE(n >= 1 && n <= 65535, "batch size must be in 1..65535 (got %d)", n);
    int rc = wvg::check_params(params);
    if (rc) return rc;
    const int L = params->levels;
    int k = 1;
    while (k < L && (1 << k) < scale) ++k;
    HIC_REQUIRE(scale == (1 << k), "scale must be 2^k with 1 <= k <= %d levels (got %d)", L, scale);
    HIC_REQUIRE(h % (1 << L) == 0 && w % (1 << L) == 0, "a scaled decode of %d levels needs multiples of %d (got %dx%d)", L,
                1 << L, h, w);
    wvg::Pyr g;
    rc = wvg::make(h, w, L, &g);
    if (rc) return rc;
    cudaStream_t st = as_stream(stream);
    const int64_t n3 = 3 * (int64_t)n, pixels = (int64_t)g.p.lh[k] * g.p.lw[k];
    double* plane[2] = {static_cast<double*>(d_work), static_cast<double*>(d_work) + wvg::plane_doubles(n, h, w)};
    int cur = (L - k) & 1;                                          // so that the last level lands in plane[0]
    HIC_LAUNCH("wavelet_approximation_load_kernel", st, wvg::approximation_load_kernel<<<wvg::blocks_for((int64_t)g.p.lh[L] * g.p.lw[L] * n3), 256, 0, st>>>(
        d_flat, g, g.p.lh[L], g.p.lw[L], (int64_t)g.p.lh[L] * g.p.lw[L], n3, plane[cur]));
    for (int l = L; l > k; --l) {                                   // the first L - k levels of the full inverse
        const int ho = g.p.lh[l], wo = g.p.lw[l];
        const int i = L - l;
        const double mul = params->multiplier * (double)(i * i + 1);
        HIC_LAUNCH("wavelet_inverse_level_kernel", st, wvg::inverse_level_kernel<<<wvg::blocks_for((int64_t)ho * wo * n3), 256, 0, st>>>(
            plane[cur], ho, wo, (int64_t)ho * wo, plane[cur ^ 1], g.p.lh[l - 1], g.p.lw[l - 1], n3, g, 1 + 3 * i, mul, d_flat));
        cur ^= 1;
    }
    // plane[cur] holds A_k, channel-planar; its (image, channel) stride is lh[k] * lw[k] = (h / scale) (w / scale)
    HIC_LAUNCH("wavelet_scaled_finish_kernel", st, wvg::scaled_finish_kernel<<<wvg::blocks_for(pixels * n), 256, 0, st>>>(
        plane[cur], pixels, pixels * n, 1.0 / scale, d_rgb_out));
    return HIC_OK;
}

int hic_wavelet_region(const int16_t* d_flat, int32_t n, int32_t h, int32_t w, const hic_wavelet_params* params, int32_t scale,
                       const int32_t* h_origin, int32_t rh, int32_t rw, void* d_work, size_t work_bytes, uint8_t* d_rgb_out,
                       void* stream) {
    using namespace hic;
    HIC_REQUIRE(d_flat && h_origin && d_work && d_rgb_out, "NULL pointer");
    HIC_REQUIRE(n >= 1 && n <= 65535, "batch size must be in 1..65535 (got %d)", n);
    int rc = wvg::check_params(params);
    if (rc) return rc;
    const int L = params->levels;
    int k = 0;
    while (k < L && (1 << k) < scale) ++k;
    HIC_REQUIRE(scale == (1 << k), "scale must be 2^k with 0 <= k <= %d levels (got %d)", L, scale);
    HIC_REQUIRE(h % (1 << L) == 0 && w % (1 << L) == 0, "a region decode of %d levels needs multiples of %d (got %dx%d)", L,
                1 << L, h, w);
    wvg::Pyr g;
    rc = wvg::make(h, w, L, &g);
    if (rc) return rc;
    HIC_REQUIRE(rh >= 1 && rw >= 1, "empty region %dx%d", rh, rw);
    const int ih = h >> k, iw = w >> k;
    for (int i = 0; i < n; ++i) {
        const int64_t top = h_origin[2 * i], left = h_origin[2 * i + 1];
        HIC_REQUIRE(top >= 0 && left >= 0 && top + rh <= ih && left + rw <= iw,
                    "region %dx%d at (%lld, %lld) is not inside the %dx%d 1/%d-scale image", rh, rw, (long long)top,
                    (long long)left, ih, iw, scale);
    }
    const size_t need = (size_t)n * 2 * sizeof(int32_t);
    HIC_REQUIRE(work_bytes >= need, "work buffer of %zu bytes is too small: %zu needed for the origins", work_bytes, need);
    HIC_REQUIRE((reinterpret_cast<uintptr_t>(d_work) & 3) == 0, "d_work must be 4-byte aligned");
    cudaStream_t st = as_stream(stream);
    HIC_CUDA(cudaMemcpyAsync(d_work, h_origin, need, cudaMemcpyHostToDevice, st));
    wvg::RegionArgs a = {reinterpret_cast<const int32_t*>(d_work), n, rh, rw, {}, 1.0 / scale};
    for (int i = 0; i < L; ++i) a.mul[i] = params->multiplier * (double)(i * i + 1);
    const int D = L - k;
    const int64_t threads = (int64_t)n * (D == 0 ? (int64_t)rh * rw : (int64_t)(rh / 2 + 1) * (rw / 2 + 1));
    HIC_REQUIRE(threads <= 256ll * INT32_MAX, "batch too large: %lld threads", (long long)threads);
    const unsigned blocks = wvg::blocks_for(threads);
    switch (D) {                     // one instantiation per number of levels to reconstruct, so the walk unrolls
#define HIC_WAVELET_REGION(d) \
        case d: HIC_LAUNCH("wavelet_region_kernel", st, wvg::region_kernel<d><<<blocks, 256, 0, st>>>(d_flat, g, a, d_rgb_out)); break;
        HIC_WAVELET_REGION(0) HIC_WAVELET_REGION(1) HIC_WAVELET_REGION(2) HIC_WAVELET_REGION(3) HIC_WAVELET_REGION(4)
        HIC_WAVELET_REGION(5)
#undef HIC_WAVELET_REGION
    }
    return HIC_OK;
}

int hic_wavelet_flat_to_bands_general(const int16_t* d_flat, int32_t n, int32_t h, int32_t w, int32_t levels, int32_t* d_bands,
                                      void* stream) {
    using namespace hic;
    HIC_REQUIRE(d_flat && d_bands, "NULL device pointer");
    HIC_REQUIRE(n >= 1, "batch size must be positive");
    wvg::Pyr g;
    const int rc = wvg::make(h, w, levels, &g);
    if (rc) return rc;
    cudaStream_t st = as_stream(stream);
    const int64_t n3 = 3 * (int64_t)n;
    HIC_LAUNCH("wavelet_flat_to_bands_kernel", st, wvg::flat_to_bands_kernel<<<wvg::blocks_for(g.p.len * n3), 256, 0, st>>>(d_flat, g, n3, d_bands));
    return HIC_OK;
}

int hic_wavelet_bands_to_flat_general(const int32_t* d_bands, int32_t n, int32_t h, int32_t w, int32_t levels, int16_t* d_flat,
                                      void* stream) {
    using namespace hic;
    HIC_REQUIRE(d_flat && d_bands, "NULL device pointer");
    HIC_REQUIRE(n >= 1, "batch size must be positive");
    wvg::Pyr g;
    const int rc = wvg::make(h, w, levels, &g);
    if (rc) return rc;
    cudaStream_t st = as_stream(stream);
    const int64_t n3 = 3 * (int64_t)n;
    HIC_CUDA(cudaMemsetAsync(d_flat, 0, (size_t)g.chan_elems * n3 * sizeof(int16_t), st));
    HIC_LAUNCH("wavelet_bands_to_flat_kernel", st, wvg::bands_to_flat_kernel<<<wvg::blocks_for(g.p.len * n3), 256, 0, st>>>(d_bands, g, n3, d_flat));
    return HIC_OK;
}

}  // extern "C"
